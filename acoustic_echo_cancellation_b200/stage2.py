"""Stage-2 residual-echo suppressor INFERENCE on the stage-1 output (the caller side of the hot path).

    LittleNetInference  <-> Little_net.forward, inference branch
                            (Stage2_lhm/scripts/network/ERB.py:252-316; used by scripts/test.py:149-169)

Three kernels of ``libaec_b200.so`` replace the module's conv-STFTs, cuDNN GRU, matmuls and transposed-conv
iSTFT: ``aec_features`` (ERB.py:254-290), ``aec_stage2_mask`` (ERB.py:293-304) and ``aec_stage2_synth``
(ERB.py:306-316).  Weights are the reference module's own ``state_dict`` (``gru1.*``, ``linear1.*``,
``linear2.*``); training stays with the reference (no autograd here).
"""
from __future__ import annotations

import ctypes as C
from typing import Mapping, Optional

import numpy as np
import torch

from . import _lib
from .spectral import batch_shift, stage2_features
from .stage1 import Stage1Config, Stage1Stream, _pair, _require_cuda_f32, _stream_ptr, num_frames, out_samples

_KEYS = {
    "gru_w_ih": ("gru1.weight_ih_l0", (96, 64)), "gru_w_hh": ("gru1.weight_hh_l0", (96, 32)),
    "gru_b_ih": ("gru1.bias_ih_l0", (96,)), "gru_b_hh": ("gru1.bias_hh_l0", (96,)),
    "lin1_w": ("linear1.weight", (32, 64)), "lin1_b": ("linear1.bias", (32,)),
    "lin2_w": ("linear2.weight", (32, 32)), "lin2_b": ("linear2.bias", (32,)),
}


def _load_weights(state_dict: Mapping[str, object], erb, device: torch.device):
    """``(weights, erb, aec_stage2_weights)``: Little_net's parameters (dots or underscores in the names) and the
    [257, 32] bank as float32 tensors on ``device``, and the C struct of their pointers."""
    w = {}
    for field, (name, shape) in _KEYS.items():
        v = state_dict.get(name, state_dict.get(name.replace(".", "_")))
        if v is None:
            raise KeyError(f"state_dict lacks {name}")
        t = torch.as_tensor(np.asarray(v) if not isinstance(v, torch.Tensor) else v).to(
            device=device, dtype=torch.float32).contiguous()
        if tuple(t.shape) != shape:
            raise ValueError(f"{name} must have shape {shape} (Little_net with 32 ERB bands)")
        w[field] = t
    erb = torch.as_tensor(np.asarray(erb) if not isinstance(erb, torch.Tensor) else erb).to(
        device=device, dtype=torch.float32).contiguous()
    if tuple(erb.shape) != (257, 32):
        raise ValueError("erb must be [257, 32]")
    return w, erb, _lib.Stage2Weights(**{k: v.data_ptr() for k, v in w.items()})


class LittleNetInference:
    """``out_wav = net(mic, ref)`` with ``net = LittleNetInference(state_dict, erb, device)``.

    ``state_dict`` maps the reference's parameter names (dots or underscores) to tensors / arrays;
    ``erb`` is the [257, 32] bank of ``EquivalentRectangularBandwidth(...).filters``."""

    def __init__(self, state_dict: Mapping[str, object], erb, device="cuda"):
        self.device = torch.device(device)
        self._w, self.erb, self._cw = _load_weights(state_dict, erb, self.device)

    def __call__(self, mic: torch.Tensor, ref: torch.Tensor, in_norm: bool = True) -> torch.Tensor:
        _require_cuda_f32("mic", mic)
        _require_cuda_f32("ref", ref)
        if mic.shape != ref.shape or mic.dim() != 2:
            raise ValueError("mic and ref must be [B, L]")
        mic, ref = mic.contiguous(), ref.contiguous()
        B, L = mic.shape
        lib = _lib.load()
        # ERB.py:254: the batch-global scalar mean/std is subtracted (torch.std is unbiased); reduced on the device
        # once per signal and passed by device pointer -- the whole forward is asynchronous, no host round trip
        shift_mic = batch_shift(mic) if in_norm else None
        shift_ref = batch_shift(ref) if in_norm else None
        feat = stage2_features(mic, ref, self.erb, in_norm=in_norm,
                               shifts=(shift_mic, shift_ref) if in_norm else None)   # [B, T, 64]
        T = num_frames(L)
        with torch.cuda.device(mic.device):
            est = torch.empty((B, T, 32), dtype=torch.float32, device=mic.device)
            out = torch.empty((B, out_samples(L)), dtype=torch.float32, device=mic.device)
            s = _stream_ptr(mic)
            _lib.check(lib.aec_stage2_mask(feat.data_ptr(), C.byref(self._cw), est.data_ptr(), B, T, 32, s),
                       "aec_stage2_mask")
            if out.numel():
                _lib.check(lib.aec_stage2_synth_dev(mic.data_ptr(), est.data_ptr(), self.erb.data_ptr(), out.data_ptr(),
                                                    B, L, L, out.shape[1], 512, 32,
                                                    shift_mic.data_ptr() if shift_mic is not None else None, s),
                           "aec_stage2_synth_dev")
        return out


def _row_mask(rows, streams: int, device) -> Optional[torch.Tensor]:
    """uint8 [streams] device mask of ``rows`` (a bool mask or stream indices), or None for all rows."""
    if rows is None:
        return None
    rows = torch.as_tensor(rows, device=device)
    if rows.dtype == torch.bool:
        mask = rows.to(torch.uint8).contiguous()
    else:
        mask = torch.zeros((streams,), dtype=torch.uint8, device=device)
        mask[rows.to(torch.int64)] = 1
    if mask.numel() != streams:
        raise ValueError("rows: a mask of one entry per stream, or stream indices")
    return mask


class Stage2Stream:
    """Online Stage 2 for ``streams`` live calls (``aec_stage2_run_stream``): ``Little_net`` with each stream's GRU
    state, last input hop and pending overlap-add half-frame kept on the device between calls.  The weights and bank
    are those of ``LittleNetInference``; there is no batch-global input shift (``in_norm=False``).

    ``process`` takes chunks of any length.  The kernel consumes whole hops of 256 samples; up to 255 samples per stream
    wait here for the next chunk, and output block g needs frame g + 1, i.e. one hop of look-ahead.  ``flush`` ends the
    listed streams: after it, a stream's concatenated output is, bit for bit, the ``(T - 1) * 256`` samples of one call
    over the whole stream (T = ``num_frames`` of its length).  ``state`` is the ``uint8 [streams, state_stride]``
    device tensor of the states (layout: include/aec_b200.h)."""

    HOP = 256
    BANDS = 32

    def __init__(self, streams: int, state_dict: Mapping[str, object], erb, device=None):
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._w, self.erb, self._cw = _load_weights(state_dict, erb, self.device)
        self._lib = _lib.load()
        self.streams = int(streams)
        self.state_bytes = int(self._lib.aec_stage2_state_bytes())
        self.state_stride = (self.state_bytes + 15) // 16 * 16
        with torch.cuda.device(self.device):
            self.state = torch.empty((self.streams, self.state_stride), dtype=torch.uint8, device=self.device)
            # pending samples, right-aligned: row b's last _npend[b] columns of mic (0) and ref (1)
            self._pend = torch.zeros((2, self.streams, self.HOP - 1), dtype=torch.float32, device=self.device)
            self._npend = torch.zeros((self.streams,), dtype=torch.int64, device=self.device)
        self.reset()

    def reset(self, rows=None):
        """Zero the state and drop the pending samples of ``rows`` (a bool mask or indices; None: all)."""
        with torch.cuda.device(self.device):
            mask = _row_mask(rows, self.streams, self.device)
            rc = self._lib.aec_stage2_state_init(self.state.data_ptr(), self.streams, self.state_stride,
                                                 mask.data_ptr() if mask is not None else None,
                                                 _stream_ptr(self.state))
            _lib.check(rc, "aec_stage2_state_init")
            if mask is None:
                self._npend.zero_()
            else:
                self._npend.masked_fill_(mask.bool(), 0)

    def state_views(self) -> dict:
        """Named views into ``state`` (writable, aliasing it): ``frames`` int64 [S], ``h`` float32 [S, 32], then
        ``mic_prev``, ``ref_prev`` and ``ola`` float32 [S, 256].  The one place on the Python side that knows the
        layout."""
        st = self.state

        def f32(off, n):
            return st[:, off:off + 4 * n].view(torch.float32)

        return {"frames": st[:, 0:8].view(torch.int64)[:, 0], "h": f32(16, 32), "mic_prev": f32(144, self.HOP),
                "ref_prev": f32(1168, self.HOP), "ola": f32(2192, self.HOP)}

    def _run(self, mic: torch.Tensor, ref: torch.Tensor, n: torch.Tensor, width: int):
        """One kernel call on left-aligned [streams, width] rows with n[b] samples each; returns ``(out, n_out)``."""
        hops = n // self.HOP
        first = (self.state_views()["frames"] == 0) & (hops > 0)      # read before the kernel advances the state
        out = torch.empty((self.streams, width), dtype=torch.float32, device=self.device)
        rc = self._lib.aec_stage2_run_stream(mic.data_ptr(), ref.data_ptr(), self.erb.data_ptr(), C.byref(self._cw),
                                             out.data_ptr(), n.data_ptr(), self.streams, width, width, width,
                                             self.state.data_ptr(), self.state_stride, self.BANDS,
                                             _stream_ptr(self.state))
        _lib.check(rc, "aec_stage2_run_stream")
        return out, (hops - first.to(torch.int64)) * self.HOP

    def process(self, mic: torch.Tensor, ref: torch.Tensor, n: Optional[torch.Tensor] = None):
        """One chunk of every stream: mic (the stage-1 error or the microphone) and ref (the far end), [streams, L]
        float32 CUDA, any L >= 0; ``n``: optional int64 [streams] device tensor, row b's chunk being its first n[b]
        samples (default L).  Returns ``out`` [streams, M] and ``n_out`` int64 [streams]: row b's new output is its first
        ``n_out[b]`` samples, zero beyond (M = the most any row can have).  Asynchronous on the current stream."""
        mic, ref = _pair(mic, ref)
        if mic.shape[0] != self.streams or mic.device != self.device:
            raise ValueError(f"mic and ref must be [{self.streams}, L] tensors on {self.device}")
        B, L = mic.shape
        H, R = self.HOP, self.HOP - 1
        width = (R + L + 3) // 4 * 4                                  # 16-byte rows
        with torch.cuda.device(self.device):
            if n is None:
                n = torch.full((B,), L, dtype=torch.int64, device=self.device)
            else:
                n = n.to(device=self.device, dtype=torch.int64).reshape(-1).clamp(0, L)
                if n.numel() != B:
                    raise ValueError("n must have one entry per stream")
            # row b: its pending samples, then the chunk; gathered from [pending (right-aligned) | chunk]
            both = torch.cat([self._pend, torch.stack([mic, ref])], dim=2)              # [2, B, R + L]
            tot = self._npend + n
            idx = (R - self._npend)[:, None] + torch.arange(width, device=self.device)[None, :]
            inp = torch.gather(both, 2, idx.clamp(max=R + L - 1).expand(2, B, width))
            inp.masked_fill_((idx >= R + L).expand(2, B, width), 0.0)
            out, n_out = self._run(inp[0], inp[1], tot, width)
            # the samples past the last whole hop wait for the next chunk
            tail = (tot - R)[:, None] + torch.arange(R, device=self.device)[None, :]
            self._pend = torch.gather(inp, 2, tail.clamp(min=0).expand(2, B, R))
            self._npend = tot % H
        return out[:, :(R + L) // H * H], n_out

    def flush(self, rows=None):
        """End the streams ``rows`` (a bool mask or indices; None: all): feed each its pending samples zero-padded to one
        hop, which yields its last block, then reset it.  Returns ``(out [streams, 256], n_out)`` like ``process``; the
        other rows get nothing and keep their state."""
        H, R = self.HOP, self.HOP - 1
        with torch.cuda.device(self.device):
            mask = _row_mask(rows, self.streams, self.device)
            j = torch.arange(H, device=self.device)[None, :]
            idx = (R - self._npend)[:, None] + j
            inp = torch.gather(self._pend, 2, idx.clamp(max=R - 1).expand(2, self.streams, H))
            inp.masked_fill_((j >= self._npend[:, None]).expand(2, self.streams, H), 0.0)
            n = torch.full((self.streams,), H, dtype=torch.int64, device=self.device)
            if mask is not None:
                n.masked_fill_(mask == 0, 0)
            out, n_out = self._run(inp[0], inp[1], n, H)
        self.reset(rows)
        return out, n_out


class AecStream:
    """The two stages online: ``Stage1Stream`` (the overlap-save filter, state carried) followed by ``Stage2Stream`` on
    (stage-1 error, far end), as ``LittleNetInference(in_norm=False)(stage1_aec(far, mic), far)`` does on whole
    signals.  The class keeps, per stream, the far-end samples stage 1 has consumed but stage 2 has not seen yet, so
    that stage 2 gets each error sample with the far-end sample it came from.

    The output lags the input by at most 255 + 256 samples: up to 255 wait in stage 1 for a whole 256-sample block, and
    a stage-2 output block needs the next hop (32 ms at 16 kHz; arithmetic, not a measurement).  ``flush`` ends streams:
    the concatenated output of a flushed stream is the whole-signal result's ``(T - 1) * 256`` samples."""

    def __init__(self, streams: int, stage1_cfg: Optional[Stage1Config], state_dict: Mapping[str, object], erb,
                 device=None):
        self.s1 = Stage1Stream(streams, stage1_cfg, device)
        self.device = self.s1.device
        self.s2 = Stage2Stream(streams, state_dict, erb, self.device)
        self.streams = self.s1.streams
        R = Stage1Stream.HOP - 1
        with torch.cuda.device(self.device):
            # far-end samples stage 1 holds back (right-aligned: row b's last _nfar[b] columns)
            self._far = torch.zeros((self.streams, R), dtype=torch.float32, device=self.device)
            self._nfar = torch.zeros((self.streams,), dtype=torch.int64, device=self.device)

    def reset(self, rows=None):
        """Restart the streams ``rows`` (a bool mask or indices; None: all) in both stages."""
        self.s1.reset(rows)
        self.s2.reset(rows)
        with torch.cuda.device(self.device):
            mask = _row_mask(rows, self.streams, self.device)
            if mask is None:
                self._nfar.zero_()
            else:
                self._nfar.masked_fill_(mask.bool(), 0)

    def process(self, far: torch.Tensor, mic: torch.Tensor):
        """One chunk of every stream: far, mic [streams, L] float32 CUDA, any L >= 0.  Returns ``(out, n_out)`` as
        ``Stage2Stream.process``."""
        far, mic = _pair(far, mic)
        B, L = far.shape
        R = Stage1Stream.HOP - 1
        err, n1 = self.s1.process(far, mic)
        with torch.cuda.device(self.device):
            # the far end from the first sample stage 1 held back: the samples its error output of this call belongs to
            tot = self._nfar + L
            idx = (R - self._nfar)[:, None] + torch.arange(R + L, device=self.device)[None, :]
            inp = torch.gather(torch.cat([self._far, far], dim=1), 1, idx.clamp(max=R + L - 1))
            far2 = inp[:, :err.shape[1]].contiguous()
            tail = (tot - R)[:, None] + torch.arange(R, device=self.device)[None, :]
            self._far = torch.gather(inp, 1, tail.clamp(min=0))
            self._nfar = tot - n1
        return self.s2.process(err, far2, n1)

    def flush(self, rows=None):
        """End the streams ``rows``: the far-end samples stage 1 still holds (their stage-1 error is zero, as
        ``stage1_aec``'s output past the last whole block) go through stage 2 with the last hop, then both stages
        restart those rows.  Returns ``(out, n_out)`` as ``Stage2Stream.flush``."""
        R = Stage1Stream.HOP - 1
        with torch.cuda.device(self.device):
            mask = _row_mask(rows, self.streams, self.device)
            j = torch.arange(R, device=self.device)[None, :]
            idx = (R - self._nfar)[:, None] + j
            f = torch.gather(self._far, 1, idx.clamp(max=R - 1))
            f.masked_fill_(j >= self._nfar[:, None], 0.0)
            n = self._nfar.clone()
            if mask is not None:
                n.masked_fill_(mask == 0, 0)
            # fewer than one hop: stage 2 only queues these samples (its own pending is empty between whole-block calls)
            self.s2.process(torch.zeros_like(f), f, n)
        out = self.s2.flush(rows)
        self.s1.reset(rows)
        with torch.cuda.device(self.device):
            if mask is None:
                self._nfar.zero_()
            else:
                self._nfar.masked_fill_(mask.bool(), 0)
        return out
