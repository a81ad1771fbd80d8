"""GPU (-m gpu): the Stage-2 and stand-alone spectral kernels (aec_spectral.cu, aec_stage2.cu) against the float64 oracle
at the launch shapes their host code selects by batch size and length.

The golden vectors pin these kernels at B = 2-3 and short lengths only.  The launch code changes shape beyond that:
  * aec_stage2_mask: 1 utterance per CTA up to B = 4 x SM count, 4 per CTA above (the last CTA partly empty unless
    B % 4 == 0);
  * aec_stage2_synth / aec_features: one CTA row per utterance, gridDim.x = 8 CTAs per utterance from B = 64, 2 from
    B = 512, each CTA walking tiles tile_i, tile_i + gridDim.x, ... (15 hops per synthesis tile, 16 frames per
    feature tile); batches above 65535 go in slices (grid.y);
  * the synthesis and analysis loads take a predicated path for rows that are not 8-byte aligned (odd L);
  * the GRU runs in chunks of 8 frames, the frame-1024 transforms in tiles of 16 frames.
Every row is compared, unless a test says otherwise.  Bars (those of the golden shapes): features and net output
2e-4 x max|ref|, STFT 2e-5 x max(1, max|ref|), iSTFT 5e-6 absolute.
"""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import acoustic_echo_cancellation_b200 as A
from acoustic_echo_cancellation_b200 import _lib
from acoustic_echo_cancellation_b200.stage1 import _disjoint_rows
from oracle import aec_oracle as O

pytestmark = pytest.mark.gpu

TOL_FEAT = 2e-4      # x max|ref|
TOL_NET = 2e-4       # x max|ref|
TOL_STFT = 2e-5      # x max(1, max|ref|)
TOL_ISTFT = 5e-6     # absolute

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _batch(spec):
    """"4sms+3" -> 4 x SM count + 3 (the launch thresholds are in units of the device's SM count); ints pass through"""
    if isinstance(spec, int):
        return spec
    k, add = spec.split("sms")
    return int(k) * _sms() + int(add or 0)


def _signals(B, L, seed):
    """mic / ref [B, L] float32 on the device: white noise of a different level per row (a row read in another row's
    place shows), with small opposite DC offsets so that the batch-global shift is not negligible"""
    g = torch.Generator(device="cuda").manual_seed(seed)
    gain = 0.1 + 0.2 * torch.rand(B, 1, device="cuda", generator=g)
    mic = gain * torch.randn(B, L, device="cuda", generator=g) + 0.01
    ref = gain.flip(0) * torch.randn(B, L, device="cuda", generator=g) - 0.02
    return mic, ref


def _weights():
    g = np.load(os.path.join(GOLDEN, "reference_stage2.npz"))
    return {k[2:]: g[k] for k in g.files if k.startswith("w_")}, g["erb"]


def _rel_err(got, want):
    assert got.shape == want.shape
    if want.size == 0:
        return 0.0
    return float(np.abs(got - want).max()) / max(float(np.abs(want).max()), 1e-30)


# B, L of each launch shape (148 SMs: 4sms = 592)
SHAPES = {
    "mask4-partial-odd-L": ("4sms+3", 12365),    # 4-warp mask, last CTA 3/4 full; per_utt 2 of 4 tiles; unaligned rows
    "mask4-partial-even-L": ("4sms+3", 12366),   # the same with every row 8-byte aligned
    "mask1-largest": ("4sms", 12365),            # the largest batch of the 1-warp mask kernel
    "per-utt-8": (100, 40013),                   # 8 CTAs per utterance, 11 synthesis / 10 feature tiles
    "single": (1, 12365),
}


@pytest.mark.parametrize("shape", list(SHAPES))
def test_little_net_matches_oracle_at_launch_shapes(shape):
    B, L = _batch(SHAPES[shape][0]), SHAPES[shape][1]
    w, erb = _weights()
    mic, ref = _signals(B, L, seed=1)
    out = A.LittleNetInference(w, erb)(mic, ref).cpu().numpy()
    want = O.stage2_little_net(mic.cpu().numpy(), ref.cpu().numpy(), erb, w)    # shift is batch-global: whole batch
    assert _rel_err(out, want) <= TOL_NET, (shape, B, L, _rel_err(out, want))


@pytest.mark.parametrize("L", [1, 255, 256, 257, 511, 512, 513, 7 * 256, 8 * 256, 9 * 256 - 1, 15 * 256, 16 * 256,
                               17 * 256 + 1])
def test_little_net_and_features_at_length_edges(L):
    """T = L // 256 + 1 frames: T = 1 (empty output, no synthesis launch), 2, 3, around the GRU chunk (T = 8, 9) and
    the synthesis tile (T = 16: 15 hops, one tile; T = 17: 16 hops, two tiles; T = 18)"""
    B = 3
    w, erb = _weights()
    mic, ref = _signals(B, L, seed=2)
    hm, hr = mic.cpu().numpy(), ref.cpu().numpy()
    out = A.LittleNetInference(w, erb)(mic, ref).cpu().numpy()
    want = O.stage2_little_net(hm, hr, erb, w)
    assert out.shape == (B, (A.num_frames(L) - 1) * 256)
    assert _rel_err(out, want) <= TOL_NET, (L, _rel_err(out, want))
    feat = A.stage2_features(mic, ref, torch.from_numpy(erb).cuda()).cpu().numpy()
    assert _rel_err(feat, O.stage2_features(hm, hr, erb)) <= TOL_FEAT


def test_little_net_without_input_normalisation():
    B, L = _batch("4sms+3"), 12365
    w, erb = _weights()
    mic, ref = _signals(B, L, seed=3)
    out = A.LittleNetInference(w, erb)(mic, ref, in_norm=False).cpu().numpy()
    want = O.stage2_little_net(mic.cpu().numpy(), ref.cpu().numpy(), erb, w, in_norm=False)
    assert _rel_err(out, want) <= TOL_NET, _rel_err(out, want)
    normed = O.stage2_little_net(mic.cpu().numpy()[:8], ref.cpu().numpy()[:8], erb, w)
    assert _rel_err(out[:8], normed) > 10 * TOL_NET           # the flag reaches the kernels: the shift is not small


def test_little_net_beyond_the_grid_y_limit():
    """65538 utterances: the synthesis (and feature) launches go in slices of 65535.  Without the batch-global shift
    the rows are independent, so the rows on both sides of the slice boundary can be checked against the oracle alone."""
    B, L = 65535 + 3, 768
    w, erb = _weights()
    mic, ref = _signals(B, L, seed=4)
    out = A.LittleNetInference(w, erb)(mic, ref, in_norm=False)
    rows = [0, 65534, 65535, B - 1]
    got = out[rows].cpu().numpy()
    want = O.stage2_little_net(mic[rows].cpu().numpy(), ref[rows].cpu().numpy(), erb, w, in_norm=False)
    assert _rel_err(got, want) <= TOL_NET, _rel_err(got, want)
    del mic, ref, out
    torch.cuda.empty_cache()


@pytest.mark.parametrize("in_norm", [True, False])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_features_match_oracle_at_launch_shapes(shape, in_norm):
    B, L = _batch(SHAPES[shape][0]), SHAPES[shape][1]
    erb = O.erb_filterbank()
    mic, ref = _signals(B, L, seed=5)
    feat = A.stage2_features(mic, ref, torch.from_numpy(erb).float().cuda(), in_norm=in_norm).cpu().numpy()
    want = O.stage2_features(mic.cpu().numpy(), ref.cpu().numpy(), erb, in_norm=in_norm)
    assert _rel_err(feat, want) <= TOL_FEAT, (shape, in_norm, _rel_err(feat, want))


@pytest.mark.parametrize("bands", [1, 17, 64])
def test_features_with_other_bank_widths(bands):
    """aec_features takes 1-64 bands; the projection loop gives band j to warp j % 4"""
    B, L = _batch("4sms+3"), 12365
    erb = O.erb_filterbank(bands=bands)
    mic, ref = _signals(B, L, seed=6)
    feat = A.stage2_features(mic, ref, torch.from_numpy(erb).float().cuda()).cpu().numpy()
    assert feat.shape == (B, A.num_frames(L), 2 * bands)
    want = O.stage2_features(mic.cpu().numpy(), ref.cpu().numpy(), erb)
    assert _rel_err(feat, want) <= TOL_FEAT, (bands, _rel_err(feat, want))


# ---- ConvSTFT / ConviSTFT -------------------------------------------------------------------------------------------
def _stft_pair(frame):
    return A.ConvSTFT(frame, frame // 2, frame, "hann", "complex"), A.ConviSTFT(frame, frame // 2, frame, "hann", "complex")


def _check_stft_istft(frame, B, L, seed):
    stft, istft = _stft_pair(frame)
    x = _signals(B, L, seed)[0]
    s = stft(x)
    want = O.stft(x.cpu().numpy(), frame, frame // 2)
    got = s.cpu().numpy()
    assert got.shape == want.shape == (B, frame + 2, A.num_frames(L, frame))
    assert float(np.abs(got - want).max()) <= TOL_STFT * max(1.0, float(np.abs(want).max()))
    y = istft(s).cpu().numpy()
    want_y = O.istft(got.astype(np.float64), frame, frame // 2)
    assert y.shape == want_y.shape
    if y.size:
        assert float(np.abs(y - want_y).max()) <= TOL_ISTFT


@pytest.mark.parametrize("frame", [512, 1024])
@pytest.mark.parametrize("L", [1, 511, 512, 513, 1023, 1024, 1025, 16 * 512 - 1, 16 * 512 + 1])
def test_stft_istft_length_edges(frame, L):
    _check_stft_istft(frame, 3, L, seed=7)


@pytest.mark.parametrize("frame", [512, 1024])
@pytest.mark.parametrize("B", [3, 70])
def test_stft_istft_several_tiles(frame, B):
    """L = 40 * 512 + 77: 41 frames at frame 1024 (3 tiles of 16), 81 at frame 512; not a multiple of the hop"""
    _check_stft_istft(frame, B, 40 * 512 + 77, seed=8)


@pytest.mark.parametrize("frame", [512, 1024])
def test_istft_of_a_free_spectrum(frame):
    """a spectrum that is no signal's STFT: non-zero imaginary parts at DC and Nyquist, which the reference's
    synthesis kernel has zero rows for"""
    K, T, B = frame // 2 + 1, 37, 5
    g = torch.Generator(device="cuda").manual_seed(9)
    spec = 0.5 * torch.randn(B, 2 * K, T, device="cuda", generator=g)
    assert bool((spec[:, K].abs() > 0).all()) and bool((spec[:, 2 * K - 1].abs() > 0).all())
    y = _stft_pair(frame)[1](spec).cpu().numpy()
    want = O.istft(spec.cpu().numpy().astype(np.float64), frame, frame // 2)
    assert y.shape == want.shape == (B, 1, (T - 1) * frame // 2)
    assert float(np.abs(y - want).max()) <= TOL_ISTFT


# ---- strided inputs --------------------------------------------------------------------------------------------------
def _views():
    """(name, view) pairs of [B, L] inputs whose rows overlap or are broadcast, and a column slice of a wider tensor"""
    g = torch.Generator(device="cuda").manual_seed(10)
    sig = 0.2 * torch.randn(40000, device="cuda", generator=g)
    wide = 0.2 * torch.randn(6, 5000, device="cuda", generator=g)
    return [("unfold", sig.unfold(0, 4096, 1000)),          # strides (1000, 1)
            ("expand", sig[:4099].expand(5, 4099)),         # strides (0, 1)
            ("column-slice", wide[:, 4:4100])]              # strides (5000, 1): disjoint rows, kept as they are


def test_strided_inputs_equal_contiguous_copies():
    views = _views()
    assert [v.stride() for _, v in views] == [(1000, 1), (0, 1), (5000, 1)]
    assert _disjoint_rows(views[2][1])[0] is views[2][1]
    for frame in (512, 1024):
        stft = _stft_pair(frame)[0]
        for name, v in views:
            assert torch.equal(stft(v), stft(v.contiguous())), (name, frame)
            assert torch.equal(stft(v[:, None]), stft(v.contiguous())), (name, frame)      # [B, 1, L] form
    for name, v in views:
        assert torch.equal(A.batch_shift(v), A.batch_shift(v.contiguous())), name
    cfg = A.Stage1Config()
    erb = torch.from_numpy(A.erb_filterbank()).float().cuda()
    for name, v in views:
        other = 0.5 * torch.roll(v.contiguous(), 7, dims=1)
        for far, mic in ((v, other), (other, v), (v, v)):   # one view, or both: far and mic share one row stride
            want = A.stage1_aec(far.contiguous(), mic.contiguous(), cfg)
            assert torch.equal(A.stage1_aec(far, mic, cfg), want), name
        err, feat = A.stage1_aec_features(v, other, erb, cfg)
        want_err, want_feat = A.stage1_aec_features(v.contiguous(), other, erb, cfg)
        assert torch.equal(err, want_err) and torch.equal(feat, want_feat), name


# ---- the by-value shift entries --------------------------------------------------------------------------------------
def test_by_value_shift_entries_equal_the_device_pointer_entries():
    """aec_features / aec_stage2_synth take the batch shift as a float (C ABI callers); with the float batch_shift
    left on the device they must give the _dev entries' bits"""
    lib = _lib.load()
    B, L = 70, 12365
    T = A.num_frames(L)
    w, erb_np = _weights()
    erb = torch.from_numpy(erb_np).cuda()
    mic, ref = _signals(B, L, seed=11)
    sm, sr = A.batch_shift(mic), A.batch_shift(ref)
    stream = int(torch.cuda.current_stream().cuda_stream)
    f_dev = torch.empty(B, T, 64, device="cuda")
    f_val = torch.empty_like(f_dev)
    _lib.check(lib.aec_features_dev(mic.data_ptr(), ref.data_ptr(), erb.data_ptr(), f_dev.data_ptr(), B, L, L, 512, 32,
                                    sm.data_ptr(), sr.data_ptr(), stream), "aec_features_dev")
    _lib.check(lib.aec_features(mic.data_ptr(), ref.data_ptr(), erb.data_ptr(), f_val.data_ptr(), B, L, L, 512, 32,
                                sm.item(), sr.item(), stream), "aec_features")
    assert torch.equal(f_dev, f_val)
    net = A.LittleNetInference(w, erb_np)
    est = torch.empty(B, T, 32, device="cuda")
    _lib.check(lib.aec_stage2_mask(f_dev.data_ptr(), C.byref(net._cw), est.data_ptr(), B, T, 32, stream), "aec_stage2_mask")
    n = (T - 1) * 256
    y_dev = torch.empty(B, n, device="cuda")
    y_val = torch.empty_like(y_dev)
    _lib.check(lib.aec_stage2_synth_dev(mic.data_ptr(), est.data_ptr(), erb.data_ptr(), y_dev.data_ptr(), B, L, L, n, 512,
                                        32, sm.data_ptr(), stream), "aec_stage2_synth_dev")
    _lib.check(lib.aec_stage2_synth(mic.data_ptr(), est.data_ptr(), erb.data_ptr(), y_val.data_ptr(), B, L, L, n, 512, 32,
                                    sm.item(), stream), "aec_stage2_synth")
    assert torch.equal(y_dev, y_val)
    assert torch.equal(y_dev, net(mic, ref))                  # ... and the wrapper is these three launches


# ---- no stray writes, run-to-run determinism -------------------------------------------------------------------------
def test_no_stray_writes_and_run_to_run_determinism():
    """canaries around every output row (output row stride wider than the row; guard regions around the dense feature
    tensor) and bitwise equality of two runs at B = 4 x SM count + 3 (a race between the warps of a CTA, or between the
    tiles a CTA walks, would show as a difference).  The inputs are ordinary in-bounds tensors."""
    lib = _lib.load()
    stream = int(torch.cuda.current_stream().cuda_stream)
    canary, pad = 12345.0, 64
    B, L = _batch("4sms+3"), 12365
    T = A.num_frames(L)
    n = (T - 1) * 256
    w, erb_np = _weights()
    erb = torch.from_numpy(erb_np).cuda()
    net = A.LittleNetInference(w, erb_np)
    mic, ref = _signals(B, L, seed=12)
    sm, sr = A.batch_shift(mic), A.batch_shift(ref)
    spec = {f: _stft_pair(f)[0](mic) for f in (512, 1024)}

    def rows_buffer(n_out):
        stride = n_out + 2 * pad + 3                          # odd: every other row starts unaligned
        return torch.full((B + 1, stride), canary, device="cuda"), stride

    def check_rows(buf, n_out):
        assert bool((buf[:B, :pad] == canary).all()) and bool((buf[:B, pad + n_out:] == canary).all())
        assert bool((buf[B] == canary).all())
        assert bool(torch.isfinite(buf[:B, pad:pad + n_out]).all())

    runs = []
    for _ in range(2):
        outs = {}
        for f in (512, 1024):
            Tf = spec[f].shape[2]
            nf = (Tf - 1) * f // 2
            buf, stride = rows_buffer(nf)
            _lib.check(lib.aec_istft(spec[f].data_ptr(), buf[0, pad:].data_ptr(), B, Tf, stride, f, stream), "aec_istft")
            torch.cuda.synchronize()
            check_rows(buf, nf)
            assert torch.equal(buf[:B, pad:pad + nf], _stft_pair(f)[1](spec[f])[:, 0])
            outs[f"istft{f}"] = buf
        fbuf = torch.full((2 * pad + B * T * 64,), canary, device="cuda")
        _lib.check(lib.aec_features_dev(mic.data_ptr(), ref.data_ptr(), erb.data_ptr(), fbuf[pad:].data_ptr(), B, L, L, 512,
                                        32, sm.data_ptr(), sr.data_ptr(), stream), "aec_features_dev")
        torch.cuda.synchronize()
        assert bool((fbuf[:pad] == canary).all()) and bool((fbuf[pad + B * T * 64:] == canary).all())
        feat = fbuf[pad:pad + B * T * 64].view(B, T, 64)
        assert bool(torch.isfinite(feat).all())
        outs["features"] = fbuf
        est = torch.empty(B, T, 32, device="cuda")
        _lib.check(lib.aec_stage2_mask(feat.data_ptr(), C.byref(net._cw), est.data_ptr(), B, T, 32, stream),
                   "aec_stage2_mask")
        buf, stride = rows_buffer(n)
        _lib.check(lib.aec_stage2_synth_dev(mic.data_ptr(), est.data_ptr(), erb.data_ptr(), buf[0, pad:].data_ptr(), B, L,
                                            L, stride, 512, 32, sm.data_ptr(), stream), "aec_stage2_synth_dev")
        torch.cuda.synchronize()
        check_rows(buf, n)
        outs["synth"] = buf
        runs.append(outs)
    for k in runs[0]:
        assert torch.equal(runs[0][k], runs[1][k]), k
    assert torch.equal(runs[0]["synth"][:B, pad:pad + n], net(mic, ref))


# ---- the fused feature epilogue of stage 1 at full occupancy ---------------------------------------------------------
def test_fused_feature_epilogue_at_full_occupancy():
    """stage1_aec_features at B = 4 x SM count + 3, 3 s: the features of 16 seeded random rows against the float64 front
    end of the error signal the kernel returned (in_norm off, so every row stands alone)"""
    B, L = _batch("4sms+3"), 48000
    g = torch.Generator(device="cuda").manual_seed(13)
    far = 0.1 * torch.randn(B, L, device="cuda", generator=g)
    mic = 0.4 * torch.roll(far, 37, dims=1) + 0.01 * torch.randn(B, L, device="cuda", generator=g)
    erb_np = A.erb_filterbank()
    err, feat = A.stage1_aec_features(far, mic, torch.from_numpy(erb_np).float().cuda())
    pick = np.sort(np.random.default_rng(13).choice(B, size=16, replace=False))
    want = O.stage2_features(err[pick].cpu().numpy(), far[pick].cpu().numpy(), erb_np, in_norm=False)
    assert _rel_err(feat[pick].cpu().numpy(), want) <= TOL_FEAT, _rel_err(feat[pick].cpu().numpy(), want)
