"""Stage-1 linear echo canceller, PyTorch-facing host API.

The reference has no stage-1 filter; this is the step a two-stage pipeline inserts between
``librosa.load`` and ``h5py.create_dataset`` in
``Stage2_lhm/generate_h5files/train_wav2h5.py:20-42``: ``(farend_speech, nearend_mic) ->
error signal`` (and, optionally, the echo estimate and per-utterance ERLE).

PyTorch is plumbing only (device memory, streams); the computation is the hand-written
sm_100a kernel behind ``aec_stage1_run`` in ``libaec_b200.so``.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import ALGO_KALMAN, ALGO_NLMS, ALGO_PBFDAF, ALGO_PBFKF  # noqa: F401  (re-exported)


@dataclass
class Stage1Config:
    """Python mirror of ``aec_cfg``.  ``frame``/``hop`` follow ``speech_conf``
    (Stage2_lhm/scripts/configs.py:1-8); ``delta=None`` means 1e-6 * frame.

    ``variant`` picks one compiled kernel build for A/B timing: ``1000 * warps_per_utterance + register cap`` (e.g.
    2168), 0 = the library default.  A build that was not compiled for (frame, partitions, algo, echo output) raises
    ``AecError`` with code -2 instead of running another one; ``stage1_aec_features`` and the frame-1024
    overlap-save filters take only ``variant=0``."""

    frame: int = 512
    partitions: int = 4
    algo: int = ALGO_NLMS
    mu: float = 0.5
    delta: Optional[float] = None
    kalman_a: float = 0.999
    kalman_lambda: float = 0.9
    kalman_c0: float = 1.0
    kalman_eps: float = 1e-10
    pb_lambda: float = 0.5
    erle_skip_hops: int = 0
    variant: int = 0
    stagger_ns: int = 0
    _c: Optional[_lib.AecCfg] = field(default=None, repr=False, compare=False)

    @property
    def hop(self) -> int:
        return self.frame // 2

    def to_c(self) -> _lib.AecCfg:
        return _lib.default_cfg(
            self.frame, partitions=self.partitions, algo=self.algo, mu=self.mu,
            delta=(1e-6 * self.frame if self.delta is None else self.delta),
            kalman_a=self.kalman_a, kalman_lambda=self.kalman_lambda, kalman_c0=self.kalman_c0,
            kalman_eps=self.kalman_eps, pb_lambda=self.pb_lambda, erle_skip_hops=self.erle_skip_hops, variant=self.variant,
            stagger_ns=self.stagger_ns)


@dataclass
class DelayConfig:
    """Python mirror of ``aec_delay_cfg``: far-end bulk-delay estimation (GCC-PHAT over the whole utterance) and the
    shift applied to the far end before stage 1.  ``max_delay`` D: largest lag searched, a power of two in [256, 8192]
    (8192 = 512 ms at 16 kHz); ``margin``: samples of echo path kept in front of the estimated delay; ``min_peak``:
    normalised correlation peak below which the far end is not shifted (DESIGN.md "Far-end delay estimation")."""

    max_delay: int = 8192
    margin: int = 128
    min_peak: float = 0.1

    def to_c(self) -> _lib.AecDelayCfg:
        c = _lib.AecDelayCfg()
        _lib.check(_lib.load().aec_delay_cfg_default(C.byref(c)), "aec_delay_cfg_default")
        c.max_delay, c.margin, c.min_peak = int(self.max_delay), int(self.margin), float(self.min_peak)
        return c


def num_frames(n_samples: int, frame: int = 512) -> int:
    """Frame count of the reference STFT (attention_ccrn.py:48-49)."""
    return int(_lib.load().aec_num_frames(int(n_samples), int(frame)))


def out_samples(n_samples: int, frame: int = 512) -> int:
    """Samples ConviSTFT returns for an ``n_samples`` input (attention_ccrn.py:99)."""
    return int(_lib.load().aec_out_samples(int(n_samples), int(frame)))


def _stream_ptr(t: torch.Tensor) -> int:
    return int(torch.cuda.current_stream(t.device).cuda_stream)


def _require_cuda_f32(name: str, t: torch.Tensor) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: acoustic_echo_cancellation_b200 has no CPU path "
                           "(use stage1_aec_host for host arrays)")
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32 (the reference stores float32 wav data)")


def _disjoint_rows(x: torch.Tensor):
    """``(x', row_stride)`` for a [B, L] tensor: ``x`` itself when its rows are unit-stride and do not overlap (a column
    slice of a wider tensor keeps its stride, no copy), else ``x.contiguous()``.  Overlapping or broadcast rows
    (``unfold`` / ``expand`` views: row stride < L) would otherwise be read as if they were ``max(stride, L)`` apart."""
    B, L = x.shape
    if x.stride(1) != 1 or (B > 1 and x.stride(0) < L):
        x = x.contiguous()
    return x, (x.stride(0) if B > 1 else L)


def _shared_rows(far: torch.Tensor, mic: torch.Tensor):
    """``(far', mic', row_stride)``: ``_disjoint_rows`` of both signals, which the stage-1 entries read with ONE row
    stride; contiguous copies of both when their strides differ."""
    far, fs = _disjoint_rows(far)
    mic, ms = _disjoint_rows(mic)
    if fs != ms:
        far, mic = far.contiguous(), mic.contiguous()
        fs = far.shape[1]
    return far, mic, fs


def _device_lengths(n_samples: Optional[torch.Tensor], B: int, device):
    """``(n_samples as a contiguous int64 CUDA tensor, its pointer)``, or ``(None, None)``."""
    if n_samples is None:
        return None, None
    n_samples = n_samples.to(device=device, dtype=torch.int64).contiguous()
    if n_samples.numel() != B:
        raise ValueError("n_samples must have B entries")
    return n_samples, n_samples.data_ptr()


def _pair(far: torch.Tensor, mic: torch.Tensor):
    _require_cuda_f32("far", far)
    _require_cuda_f32("mic", mic)
    if far.dim() == 1:
        far, mic = far[None], mic[None]
    if far.shape != mic.shape or far.dim() != 2 or far.device != mic.device:
        raise ValueError("far and mic must be [B, L] tensors of equal shape on one device")
    return far, mic


def estimate_delay(far: torch.Tensor, mic: torch.Tensor, cfg: Optional[DelayConfig] = None,
                   n_samples: Optional[torch.Tensor] = None, return_corr: bool = False):
    """Far-end bulk delay of every utterance (``aec_delay_estimate``): GCC-PHAT of ``mic`` against ``far`` at lags
    0 .. ``cfg.max_delay``.

    far, mic : [B, L] float32 CUDA;  n_samples: optional int64 [B] true lengths.
    Returns CUDA tensors ``(delay int32 [B], shift int32 [B], peak float32 [B])``, plus ``corr`` [B, D + 1] (the
    normalised correlation r) with ``return_corr``.  ``shift`` is what ``align_far`` delays the far end by.
    Asynchronous on the current stream of ``far.device``."""
    cfg = cfg or DelayConfig()
    far, mic = _pair(far, mic)
    far, mic, in_stride = _shared_rows(far, mic)
    B, L = far.shape
    c = cfg.to_c()
    with torch.cuda.device(far.device):
        delay = torch.empty((B,), dtype=torch.int32, device=far.device)
        shift = torch.empty_like(delay)
        peak = torch.empty((B,), dtype=torch.float32, device=far.device)
        corr = torch.empty((B, int(cfg.max_delay) + 1), dtype=torch.float32, device=far.device) if return_corr else None
        n_samples, ns_ptr = _device_lengths(n_samples, B, far.device)
        rc = _lib.load().aec_delay_estimate(far.data_ptr(), mic.data_ptr(), ns_ptr, B, L, in_stride, C.byref(c),
                                            delay.data_ptr(), shift.data_ptr(), peak.data_ptr(),
                                            corr.data_ptr() if corr is not None else None, _stream_ptr(far))
        _lib.check(rc, "aec_delay_estimate")
    return (delay, shift, peak, corr) if return_corr else (delay, shift, peak)


def align_far(far: torch.Tensor, shift: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``out[b, n] = far[b, n - shift[b]]`` for ``n >= shift[b]``, 0 below (``aec_delay_align``); rows keep their
    length L.  far: [B, L] float32 CUDA; shift: int [B] (``estimate_delay``'s, or any).  ``out`` must not overlap far."""
    _require_cuda_f32("far", far)
    squeeze = far.dim() == 1
    if squeeze:
        far = far[None]
    if far.dim() != 2:
        raise ValueError("far must be a [B, L] tensor")
    far, in_stride = _disjoint_rows(far)
    B, L = far.shape
    shift = shift.to(device=far.device, dtype=torch.int32).reshape(-1).contiguous()
    if shift.numel() != B:
        raise ValueError("shift must have B entries")
    with torch.cuda.device(far.device):
        if out is None:
            out = torch.empty((B, L), dtype=torch.float32, device=far.device)
        else:
            if squeeze and out.dim() == 1:
                out = out[None]
            if out.shape != (B, L) or not out.is_cuda or out.dtype != torch.float32 or out.stride(1) != 1 \
                    or (B > 1 and out.stride(0) < L):
                raise ValueError("out must be a [B, L] float32 CUDA tensor with disjoint unit-stride rows")
        out_stride = out.stride(0) if B > 1 else max(out.stride(0), L)
        rc = _lib.load().aec_delay_align(far.data_ptr(), out.data_ptr(), shift.data_ptr(), B, L, in_stride, out_stride,
                                         _stream_ptr(far))
        _lib.check(rc, "aec_delay_align")
    return out[0] if squeeze else out


def stage1_aec(far: torch.Tensor, mic: torch.Tensor, cfg: Optional[Stage1Config] = None,
               n_samples: Optional[torch.Tensor] = None, return_echo: bool = False,
               return_erle: bool = False, out: Optional[torch.Tensor] = None,
               align: Optional[DelayConfig] = None, return_shift: bool = False):
    """Run the stage-1 canceller on a batch of CUDA tensors.

    far, mic : [B, L] float32 CUDA (``farend_speech`` / ``nearend_mic`` rows)
    n_samples: optional int64 [B] true lengths (ragged batch, zero-padded to L as the
               reference's ``collate_fn`` does, Stage2_lhm/scripts/train1.py:52-61)
    align    : optional ``DelayConfig``: estimate each utterance's far-end delay and run stage 1 on the far end
               delayed by the resulting shift (``estimate_delay`` + ``align_far`` into a temporary buffer); off by
               default.  ``return_shift`` (needs ``align``) also returns that shift, int32 [B].
    Returns ``err`` [B, L] (zero beyond ``out_samples(n_b)``), plus ``echo`` [B, L], ``erle_db`` [B] and
    ``shift`` [B] when requested (in that order).
    The call is asynchronous on the current stream of ``far.device``.
    """
    cfg = cfg or Stage1Config()
    if return_shift and align is None:
        raise ValueError("return_shift needs align")
    far, mic = _pair(far, mic)
    shift = None
    if align is not None:
        _, shift, _ = estimate_delay(far, mic, align, n_samples)
        mic, m_stride = _disjoint_rows(mic)
        with torch.cuda.device(far.device):
            buf = torch.empty((far.shape[0], m_stride), dtype=torch.float32, device=far.device)
        far = align_far(far, shift, out=buf[:, :far.shape[1]])      # rows spaced like mic's: no copy of mic below
    far, mic, in_stride = _shared_rows(far, mic)
    B, L = far.shape
    lib = _lib.load()
    with torch.cuda.device(far.device):
        if out is None:
            out = torch.empty((B, L), dtype=torch.float32, device=far.device)
        elif out.shape != (B, L) or not out.is_cuda or out.dtype != torch.float32 or out.stride(1) != 1:
            raise ValueError("out must be a [B, L] float32 CUDA tensor with unit inner stride")
        echo = torch.empty_like(out) if return_echo else None
        erle = torch.empty((B,), dtype=torch.float32, device=far.device) if return_erle else None
        n_samples, ns_ptr = _device_lengths(n_samples, B, far.device)
        out_stride = out.stride(0) if B > 1 else max(out.stride(0), L)
        if echo is not None and echo.stride(0) != out.stride(0):
            echo = torch.empty_strided(out.shape, out.stride(), dtype=torch.float32, device=far.device)
        c = cfg.to_c()
        rc = lib.aec_stage1_run(far.data_ptr(), mic.data_ptr(), out.data_ptr(),
                                echo.data_ptr() if echo is not None else None,
                                erle.data_ptr() if erle is not None else None,
                                ns_ptr, B, L, in_stride, out_stride, C.byref(c), _stream_ptr(far))
        _lib.check(rc, "aec_stage1_run")
    res = [out]
    if return_echo:
        res.append(echo)
    if return_erle:
        res.append(erle)
    if return_shift:
        res.append(shift)
    return res[0] if len(res) == 1 else tuple(res)


def stage1_aec_features(far: torch.Tensor, mic: torch.Tensor, erb: torch.Tensor, cfg: Optional[Stage1Config] = None,
                        n_samples: Optional[torch.Tensor] = None, return_erle: bool = False,
                        out: Optional[torch.Tensor] = None):
    """Stage 1 with the Stage-2 feature front end fused into the kernel (``aec_stage1_run_features``).

    Returns ``(err [B, L], feat [B, T, 64])`` (+ ``erle_db [B]``): ``feat`` is what
    ``stage2_features(err, far, erb, in_norm=False)`` gives -- ``cat[err_erb, |err_erb - far_erb|]`` of
    Little_net.forward (Stage2_lhm/scripts/network/ERB.py:262-290) with the stage-1 error in the microphone's place --
    without re-reading ``err`` and ``far`` from HBM and without a second far-end STFT.  ``erb``: [257, 32] float32 CUDA."""
    cfg = cfg or Stage1Config()
    _require_cuda_f32("far", far)
    _require_cuda_f32("mic", mic)
    _require_cuda_f32("erb", erb)
    if far.dim() == 1:
        far, mic = far[None], mic[None]
    if far.shape != mic.shape or far.dim() != 2 or far.device != mic.device:
        raise ValueError("far and mic must be [B, L] tensors of equal shape on one device")
    if tuple(erb.shape) != (257, 32):
        raise ValueError("erb must be [257, 32]")
    key = (erb.data_ptr(), erb._version)
    if key not in _checked_banks:
        nz = erb != 0
        idx = torch.arange(257, device=erb.device)[:, None].expand(257, 32)
        span = torch.where(nz, idx, torch.full_like(idx, -1)).amax(0) - torch.where(nz, idx, torch.full_like(idx, 10 ** 6)).amin(0) + 1
        if int(span.clamp(min=0).sum()) > 512:
            raise ValueError("the ERB bank has more than 512 coefficients inside its bands' non-zero ranges")
        _checked_banks.add(key)
    far, mic, in_stride = _shared_rows(far, mic)
    erb = erb.contiguous()
    B, L = far.shape
    lib = _lib.load()
    with torch.cuda.device(far.device):
        if out is None:
            out = torch.empty((B, L), dtype=torch.float32, device=far.device)
        elif out.shape != (B, L) or not out.is_cuda or out.dtype != torch.float32 or out.stride(1) != 1:
            raise ValueError("out must be a [B, L] float32 CUDA tensor with unit inner stride")
        feat = torch.empty((B, num_frames(L, cfg.frame), 64), dtype=torch.float32, device=far.device)
        erle = torch.empty((B,), dtype=torch.float32, device=far.device) if return_erle else None
        ns_ptr = None
        if n_samples is not None:
            n_samples = n_samples.to(device=far.device, dtype=torch.int64).contiguous()
            if n_samples.numel() != B:
                raise ValueError("n_samples must have B entries")
            ns_ptr = n_samples.data_ptr()
        out_stride = out.stride(0) if B > 1 else max(out.stride(0), L)
        c = cfg.to_c()
        rc = lib.aec_stage1_run_features(far.data_ptr(), mic.data_ptr(), out.data_ptr(),
                                         erle.data_ptr() if erle is not None else None, feat.data_ptr(), erb.data_ptr(),
                                         ns_ptr, B, L, in_stride, out_stride, C.byref(c), _stream_ptr(far))
        _lib.check(rc, "aec_stage1_run_features")
    return (out, feat, erle) if return_erle else (out, feat)


_checked_banks = set()


class Stage1Stream:
    """Online stage 1 for ``streams`` live calls (``aec_stage1_run_stream``): the frame-512 overlap-save filters
    (algo 2 / 3) with each stream's filter state kept on the device between calls, so that a chunk continues where the
    previous one stopped.  Chunked processing gives bit for bit the output of ``stage1_aec`` over the whole signal.

    ``process`` takes chunks of any length.  The kernel consumes whole blocks of 256 samples; up to 255 samples per
    stream wait here for the next chunk, so the output lags the input by at most one block (16 ms at 16 kHz).
    ``state`` is the ``uint8 [streams, state_stride]`` device tensor of the states (layout: include/aec_b200.h)."""

    HOP = 256

    def __init__(self, streams: int, cfg: Optional[Stage1Config] = None, device=None):
        self.cfg = cfg or Stage1Config(algo=ALGO_PBFDAF)
        self._c = self.cfg.to_c()
        self._lib = _lib.load()
        nbytes = int(self._lib.aec_stage1_state_bytes(C.byref(self._c)))
        _lib.check(min(nbytes, 0), "aec_stage1_state_bytes")
        self.streams = int(streams)
        self.state_bytes = nbytes
        self.state_stride = (nbytes + 15) // 16 * 16
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        with torch.cuda.device(self.device):
            self.state = torch.empty((self.streams, self.state_stride), dtype=torch.uint8, device=self.device)
            # pending samples, right-aligned: row b's last _npend[b] columns
            self._pend = torch.zeros((2, self.streams, self.HOP - 1), dtype=torch.float32, device=self.device)
            self._npend = torch.zeros((self.streams,), dtype=torch.int64, device=self.device)
        self.reset()

    def reset(self, rows=None):
        """Re-initialise the filter state and drop the pending samples of ``rows`` (a bool mask or indices; None: all)."""
        mask = None
        with torch.cuda.device(self.device):
            if rows is not None:
                rows = torch.as_tensor(rows, device=self.device)
                if rows.dtype == torch.bool:
                    mask = rows.to(torch.uint8).contiguous()
                else:
                    mask = torch.zeros((self.streams,), dtype=torch.uint8, device=self.device)
                    mask[rows.to(torch.int64)] = 1
                if mask.numel() != self.streams:
                    raise ValueError("rows: a mask of one entry per stream, or stream indices")
            rc = self._lib.aec_stage1_state_init(self.state.data_ptr(), self.streams, self.state_stride,
                                                 mask.data_ptr() if mask is not None else None, C.byref(self._c),
                                                 _stream_ptr(self.state))
            _lib.check(rc, "aec_stage1_state_init")
            if mask is None:
                self._npend.zero_()
            else:
                self._npend.masked_fill_(mask.bool(), 0)

    def state_views(self) -> dict:
        """Named views into ``state`` (writable, aliasing it): ``blocks`` int64 [S], ``prev`` float32 [S, 256], ``W`` and
        ``X`` complex64 [S, P, 257], then ``Pw`` float32 [S, 257] (algo 2) or ``Psi`` [S, 257] and ``C`` [S, P, 257]
        (algo 3).  The one place on the Python side that knows the layout."""
        P, K = self.cfg.partitions, 257
        a16 = lambda n: (n + 15) // 16 * 16       # noqa: E731
        w0 = 16 + 4 * self.HOP
        x0 = w0 + a16(8 * P * K)
        s0 = x0 + a16(8 * P * K)
        c0 = s0 + a16(4 * K)
        st = self.state

        def f32(off, n):
            return st[:, off:off + 4 * n].view(torch.float32)

        v = {"blocks": st[:, 0:8].view(torch.int64)[:, 0],
             "prev": f32(16, self.HOP),
             "W": st[:, w0:w0 + 8 * P * K].view(torch.complex64).unflatten(1, (P, K)),
             "X": st[:, x0:x0 + 8 * P * K].view(torch.complex64).unflatten(1, (P, K))}
        if self.cfg.algo == ALGO_PBFKF:
            v["Psi"] = f32(s0, K)
            v["C"] = f32(c0, P * K).unflatten(1, (P, K))
        else:
            v["Pw"] = f32(s0, K)
        return v

    def process(self, far: torch.Tensor, mic: torch.Tensor, return_echo: bool = False, return_erle: bool = False):
        """One chunk of every stream: far, mic [streams, L] float32 CUDA, any L >= 0.  Returns ``err`` [streams, M] and
        ``n_out`` int64 [streams] (M = the most whole-block samples any row can have; row b's output is its first
        ``n_out[b]`` samples, zero beyond), then ``echo`` [streams, M] and ``erle_db`` [streams] (over this call's blocks
        from ``erle_skip_hops`` blocks into the stream) when asked for.  Asynchronous on the current stream."""
        far, mic = _pair(far, mic)
        if far.shape[0] != self.streams or far.device != self.device:
            raise ValueError(f"far and mic must be [{self.streams}, L] tensors on {self.device}")
        B, L = far.shape
        H, R = self.HOP, self.HOP - 1
        width = (R + L + 3) // 4 * 4                                  # 16-byte rows: the bulk-copy staging path
        M = (R + L) // H * H
        with torch.cuda.device(self.device):
            # row b: its pending samples, then the chunk; gathered from [pending (right-aligned) | chunk]
            both = torch.cat([self._pend, torch.stack([far, mic])], dim=2)                # [2, B, R + L]
            n = self._npend + L
            idx = (R - self._npend)[:, None] + torch.arange(width, device=self.device)[None, :]
            inp = torch.gather(both, 2, idx.clamp(max=R + L - 1).expand(2, B, width))
            inp.masked_fill_((idx >= R + L).expand(2, B, width), 0.0)
            n_out = n // H * H
            err = torch.empty((B, width), dtype=torch.float32, device=self.device)
            echo = torch.empty_like(err) if return_echo else None
            erle = torch.empty((B,), dtype=torch.float32, device=self.device) if return_erle else None
            rc = self._lib.aec_stage1_run_stream(inp[0].data_ptr(), inp[1].data_ptr(), err.data_ptr(),
                                                 echo.data_ptr() if echo is not None else None,
                                                 erle.data_ptr() if erle is not None else None,
                                                 n.data_ptr(), B, width, width, width, C.byref(self._c),
                                                 self.state.data_ptr(), self.state_stride, _stream_ptr(far))
            _lib.check(rc, "aec_stage1_run_stream")
            # the samples past the last whole block wait for the next chunk
            tail = (n - R)[:, None] + torch.arange(R, device=self.device)[None, :]
            self._pend = torch.gather(inp, 2, tail.clamp(min=0).expand(2, B, R))
            self._npend = n - n_out
        res = [err[:, :M], n_out]
        if return_echo:
            res.append(echo[:, :M])
        if return_erle:
            res.append(erle)
        return tuple(res)


class HostPipeline:
    """Host-buffer entry (``aec_stage1_run_host``; ``aec_stage1_run_host_pcm16`` for int16 PCM inputs,
    scaled by 1/32768 on the GPU): numpy arrays in, numpy arrays out, copies pipelined against the kernel
    in slices.  This is the call a ``create_h5``-style data-prep
    loop makes (Stage2_lhm/generate_h5files/train_wav2h5.py:20-42)."""

    def __init__(self, slice_utterances: int, max_samples: int, device: int = 0, slots: int = 0,
                 ramp: bool = True):
        """``slots``: slices in flight (0 = library default, 4); ``ramp``: grow the first slices from 16
        utterances so that the first download starts early.  One context per thread: a pipeline is not
        re-entrant (include/aec_b200.h)."""
        self.device = device
        self._ctx = C.c_void_p()
        self._lib = _lib.load()
        with torch.cuda.device(device):
            _lib.check(self._lib.aec_host_ctx_create_ex(C.byref(self._ctx), int(slice_utterances), int(max_samples),
                                                        int(slots), 0 if ramp else 1), "aec_host_ctx_create_ex")
        self.max_samples = int(max_samples)
        self.slice_utterances = int(slice_utterances)

    def close(self):
        if self._ctx:
            with torch.cuda.device(self.device):
                self._lib.aec_host_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def wait(self):
        """Complete every deferred ``run(..., wait=False)`` call: their outputs are in host memory afterwards."""
        with torch.cuda.device(self.device):
            _lib.check(self._lib.aec_host_ctx_wait(self._ctx), "aec_host_ctx_wait")
        self._keep = []

    def run(self, far: np.ndarray, mic: np.ndarray, cfg: Optional[Stage1Config] = None,
            n_samples: Optional[np.ndarray] = None, err: Optional[np.ndarray] = None,
            echo: Optional[np.ndarray] = None, erle: Optional[np.ndarray] = None, wait: bool = True,
            align: Optional[DelayConfig] = None, shift: Optional[np.ndarray] = None,
            peak: Optional[np.ndarray] = None):
        """``wait=False`` (streaming, batch after batch): return once the last slice is enqueued, so that the tail of
        this batch runs under the first uploads of the next; outputs are complete after ``wait()``.  Consecutive
        deferred calls need different output arrays.  ``align``: estimate each utterance's far-end delay and run
        stage 1 on the shifted far end (``aec_stage1_run_host_ex``); ``shift`` (int32 [B]) and ``peak`` (float32 [B])
        receive the estimator's outputs, like ``erle``."""
        cfg = cfg or Stage1Config()
        pcm16 = far.dtype == np.int16
        item = 2 if pcm16 else 4
        for name, a in (("far", far), ("mic", mic)):
            if a.dtype != far.dtype or a.dtype not in (np.float32, np.int16) or a.ndim != 2 or a.strides[1] != item:
                raise TypeError(f"{name} must be a 2-D float32 (or int16 PCM) array with contiguous rows")
        if far.shape != mic.shape or far.strides[0] != mic.strides[0]:
            raise ValueError("far and mic must share shape and row stride")
        B, L = far.shape
        if err is None:
            err = np.empty((B, L), dtype=np.float32)
        for name, a in (("err", err), ("echo", echo)):
            if a is not None and (a.dtype != np.float32 or a.shape != (B, L) or a.strides[1] != 4):
                raise TypeError(f"{name} must be a [B, L] float32 array with contiguous rows")
        if echo is not None and echo.strides[0] != err.strides[0]:
            raise ValueError("echo and err must share the row stride")
        for name, a, dt in (("shift", shift, np.int32), ("peak", peak, np.float32)):
            if a is not None and (a.dtype != dt or a.shape != (B,) or not a.flags.c_contiguous):
                raise TypeError(f"{name} must be a contiguous {np.dtype(dt).name} array of B entries")
        if align is None and (shift is not None or peak is not None):
            raise ValueError("shift / peak need align")
        ns = None
        if n_samples is not None:
            ns = np.ascontiguousarray(n_samples, dtype=np.int64)
        c = cfg.to_c()
        dc = align.to_c() if align is not None else None
        fn = self._lib.aec_stage1_run_host_pcm16_ex if pcm16 else self._lib.aec_stage1_run_host_ex
        if not wait:     # the arrays of a deferred call must outlive it
            self._keep = getattr(self, "_keep", [])[-8:] + [(far, mic, err, echo, erle, ns, shift, peak)]
        with torch.cuda.device(self.device):
            _lib.check(self._lib.aec_host_ctx_set_deferred(self._ctx, 0 if wait else 1), "aec_host_ctx_set_deferred")
            rc = fn(self._ctx, far.ctypes.data, mic.ctypes.data, err.ctypes.data,
                    echo.ctypes.data if echo is not None else None,
                    erle.ctypes.data if erle is not None else None,
                    ns.ctypes.data if ns is not None else None,
                    B, L, far.strides[0] // item, err.strides[0] // 4, C.byref(c),
                    C.byref(dc) if dc is not None else None,
                    shift.ctypes.data if shift is not None else None,
                    peak.ctypes.data if peak is not None else None)
        _lib.check(rc, "aec_stage1_run_host_pcm16_ex" if pcm16 else "aec_stage1_run_host_ex")
        return err


class _PinnedBlock:
    """Owner of one ``aec_host_alloc_ex`` allocation; freed when the last numpy view of it dies."""

    def __init__(self, nbytes: int, flags: int):
        self.ptr = C.c_void_p()
        self._lib = _lib.load()
        _lib.check(self._lib.aec_host_alloc_ex(C.byref(self.ptr), int(nbytes), int(flags)), "aec_host_alloc_ex")
        self.nbytes = int(nbytes)

    def __del__(self):
        try:
            if self.ptr:
                self._lib.aec_host_free(self.ptr)
                self.ptr = C.c_void_p()
        except Exception:
            pass


HOST_WRITE_COMBINED = 1
HOST_PORTABLE = 2


def pinned_empty(shape, dtype=np.float32, flags: int = 0) -> np.ndarray:
    """numpy array in page-locked host memory (``aec_host_alloc_ex``: cudaHostAlloc).  ``flags``:
    ``HOST_WRITE_COMBINED`` for buffers the CPU only writes (inputs), ``HOST_PORTABLE``."""
    shape = tuple(int(x) for x in shape)
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) if shape else 1
    block = _PinnedBlock(max(n * dt.itemsize, 1), flags)
    buf = (C.c_char * block.nbytes).from_address(block.ptr.value)
    buf._aec_owner = block            # keeps the allocation alive as long as any view of `buf` is
    return np.frombuffer(buf, dtype=dt, count=n).reshape(shape)


def is_pinned(a: np.ndarray) -> bool:
    """True if the array's memory is page-locked host memory known to CUDA (``aec_host_is_pinned``)."""
    return int(_lib.load().aec_host_is_pinned(a.ctypes.data)) == 1


def fp32_peak_tflops(iters: int = 4096) -> float:
    """Measured dependent-free FFMA throughput of the current device (roofline denominator)."""
    v = C.c_double(0.0)
    _lib.check(_lib.load().aec_bench_fp32_peak(int(iters), C.byref(v),
                                               int(torch.cuda.current_stream().cuda_stream)), "aec_bench_fp32_peak")
    return float(v.value)


def launch_count(reset: bool = False) -> int:
    return int(_lib.load().aec_launch_count(1 if reset else 0))
