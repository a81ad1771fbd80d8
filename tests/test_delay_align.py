"""Far-end delay estimation and alignment (aec_delay_estimate / aec_delay_align, DelayConfig, stage1_aec(align=...),
HostPipeline.run(align=...), the generators' --stage1_align_max_delay).

CPU: the float64 oracle (oracle/delay_oracle.py) against the direct correlation sum and on synth signals with a bulk
delay, the ERLE gain of alignment through the stage-1 oracle, the float32 drift of the GPU test rows, synth's
bulk_delay=0 signals, argument errors and the generators' extra dataset.
GPU: the kernels against the float64 oracle on every row, launch shapes, batch invariance, determinism, canaries, the
end-to-end paths."""
import ctypes as C
import os
import types

import numpy as np
import pytest
from scipy.signal import fftconvolve

import acoustic_echo_cancellation_b200 as A
from acoustic_echo_cancellation_b200 import _lib, synth, wav2h5
from oracle import aec_oracle as O
from oracle import delay_oracle as DO

CORR_TOL = 1e-4
DELAYS = (0, 1, 255, 256, 700, 3200)        # + D - 30
LEVELS = (1.0, 1e-2, 1e-3, 3e-5)


# ------------------------------------------------------------------------------------------
# test rows (shared by the CPU drift check and the GPU comparison)
# ------------------------------------------------------------------------------------------
def _rows(D: int):
    """(far [B, L], mic [B, L], n [B], names): bulk delays x single / double talk, ragged lengths (noise beyond n),
    one utterance at four levels, a silent far end, and a constant pair whose block products are DC only."""
    L = 2 * D + 6000
    far, mic, n, names = [], [], [], []

    def add(f, m, nb, name):
        far.append(np.asarray(f, np.float32))
        mic.append(np.asarray(m, np.float32))
        n.append(nb)
        names.append(name)

    for i, d in enumerate(DELAYS + (D - 30,)):
        for dt in (False, True):
            u = synth.make_utterance(100 + i, L, rir_len=512, double_talk=dt, bulk_delay=d)
            add(u["far"], u["mic"], L, f"d{d}{'_dt' if dt else ''}")
    rng = np.random.default_rng(7)
    u = synth.make_utterance(120, L, rir_len=512, bulk_delay=min(300, D - 100))
    for nb in (0, 1, D - 1, D, D + 1, 2 * D + 1, L):
        f, m = u["far"].copy(), u["mic"].copy()
        f[nb:] = rng.standard_normal(L - nb)          # must not be read
        m[nb:] = rng.standard_normal(L - nb)
        add(f, m, nb, f"n{nb}")
    u = synth.make_utterance(130, L, rir_len=512, bulk_delay=min(500, D // 2))
    for lv in LEVELS:
        add(u["far"] * np.float32(lv), u["mic"] * np.float32(lv), L, f"level{lv:g}")
    add(np.zeros(L), u["mic"], L, "silent_far")
    # far constant, mic constant from sample D on, n a multiple of D: every block product Y_s conj(X_s) is DC only
    nd = (L // D) * D
    m = np.zeros(L)
    m[D:] = 0.25
    add(np.full(L, 0.5), m, nd, "dc_only")
    return np.stack(far), np.stack(mic), np.array(n, np.int64), names


_ORACLE = {}


def _oracle(D: int):
    if D not in _ORACLE:
        far, mic, n, names = _rows(D)
        cfg = DO.DelayConfig(max_delay=D)
        _ORACLE[D] = (far, mic, n, names, DO.estimate(far, mic, cfg, n), DO.estimate(far, mic, cfg, n, np.float32))
    return _ORACLE[D]


# ------------------------------------------------------------------------------------------
# CPU: oracle
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [256, 2048])
def test_oracle_cross_spectrum_is_the_linear_correlation(D):
    rng = np.random.default_rng(D)
    for n in (1, D - 1, D, D + 1, 3 * D + 5):
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        r = np.fft.irfft(DO.cross_spectrum(x, y, D), 2 * D)[:D + 1]
        ref = DO.linear_xcorr(x, y, D)
        assert np.abs(r - ref).max() <= 1e-9 * np.abs(ref).max(), n


def test_oracle_recovers_the_bulk_delay_of_synth_signals():
    """the estimate moves with the bulk delay sample for sample and lies on the response's first taps, in single talk
    and in double talk"""
    for dt in (False, True):
        for u in range(3):
            base = int(DO.estimate(synth.make_utterance(u, 160000, double_talk=dt)["far"][None],
                                   synth.make_utterance(u, 160000, double_talk=dt)["mic"][None])["delay"][0])
            assert 0 <= base < 64
            for d in (500, 3200, 7000):
                s = synth.make_utterance(u, 160000, double_talk=dt, bulk_delay=d)
                e = DO.estimate(s["far"], s["mic"])
                assert int(e["delay"][0]) == d + base, (dt, u, d)
                assert 0.15 <= e["peak"][0] <= 1.0
                assert int(e["shift"][0]) == d + base - 128


def test_oracle_unrelated_signals_stay_below_the_threshold():
    for u in range(4):
        a = synth.make_utterance(u, 160000)
        b = synth.make_utterance(u + 50, 160000, double_talk=True)
        e = DO.estimate(a["far"], b["mic"])
        assert e["peak"][0] < 0.1 and e["shift"][0] == 0


def _erle_second_half(mic, err):
    m = err.shape[-1]
    return float(O.erle_db(mic[None, m // 2:m], err[None, m // 2:])[0])


def test_oracle_alignment_restores_the_overlap_save_filter():
    """6 s at 16 kHz, 200 ms bulk delay, overlap-save NLMS (algo 2), P = 4: the filter makes the echo worse
    unaligned and is back at the noise floor aligned"""
    u = synth.make_utterance(0, 96000, bulk_delay=3200)
    e = DO.estimate(u["far"], u["mic"])
    cfg = O.AecConfig(partitions=4, algo=O.ALGO_PBFDAF)
    plain = O.stage1(u["far"][None], u["mic"][None], cfg)["err"][0]
    aligned = O.stage1(DO.align(u["far"], e["shift"]), u["mic"][None], cfg)["err"][0]
    assert _erle_second_half(u["mic"], plain) < 0.0
    assert _erle_second_half(u["mic"], aligned) >= 35.0


def test_oracle_align_definition():
    far = np.arange(1, 11, dtype=np.float32)[None].repeat(4, 0)
    out = DO.align(far, [0, 3, 10, 99])
    assert np.array_equal(out[0], far[0])
    assert np.array_equal(out[1], np.r_[0, 0, 0, far[1, :7]])
    assert not out[2].any() and not out[3].any()


@pytest.mark.parametrize("D", [256, 2048, 8192])
def test_gpu_rows_are_well_conditioned_in_float32(D):
    """float32 rounding alone moves corr by at least 10x less than the GPU tolerance on every test row, and the
    null rows are exactly null"""
    far, mic, n, names, ref, r32 = _oracle(D)
    drift = np.abs(r32["corr"] - ref["corr"]).max(axis=1)
    assert drift.max() <= CORR_TOL / 10, dict(zip(names, drift))
    for name in ("silent_far", "dc_only", "n0"):
        i = names.index(name)
        assert ref["delay"][i] == 0 and ref["peak"][i] == 0 and ref["shift"][i] == 0 and not ref["corr"][i].any()


def test_synth_bulk_delay_zero_is_the_existing_signal():
    """bulk_delay=0 gives the signals the generator gave before it had the parameter (formula restated here)"""
    for dt in (False, True):
        u = synth.make_utterance(5, 7000, rir_len=512, double_talk=dt)
        v = synth.make_utterance(5, 7000, rir_len=512, double_talk=dt, bulk_delay=0)
        for k in u:
            assert np.array_equal(u[k], v[k])
        far = synth._speechlike(np.random.default_rng(1005), 7000, 16000)
        echo = fftconvolve(far, synth.make_rir(5, 512))[:7000]
        assert np.array_equal(u["far"], far.astype(np.float32))
        if not dt:
            noise = np.random.default_rng(4005).standard_normal(7000) * np.sqrt((echo ** 2).mean()) * 10.0 ** -2
            assert np.array_equal(u["mic"], (echo + noise).astype(np.float32))
    b = synth.make_batch(3, 2, 5000, rir_len=256, double_talk=True)
    c = synth.make_batch(3, 2, 5000, rir_len=256, double_talk=True, bulk_delay=0)
    assert all(np.array_equal(b[k], c[k]) for k in b)
    d = synth.make_utterance(5, 7000, rir_len=512, bulk_delay=40)
    assert np.abs(d["echo"][:40]).max() < 1e-12 < np.abs(d["echo"][40:]).max()       # (fftconvolve rounding)


# ------------------------------------------------------------------------------------------
# CPU: C ABI and generators
# ------------------------------------------------------------------------------------------
def test_delay_cfg_default_and_layout():
    assert C.sizeof(_lib.AecDelayCfg) == 32
    c = A.DelayConfig().to_c()
    assert (c.max_delay, c.margin) == (8192, 128) and c.min_peak == pytest.approx(0.1)
    assert _lib.load().aec_delay_cfg_default(None) == -1


def test_delay_argument_errors_do_not_need_a_gpu():
    lib = _lib.load()
    f = np.zeros(64, dtype=np.float32).ctypes.data
    i = np.zeros(64, dtype=np.int32).ctypes.data
    est = lib.aec_delay_estimate

    def cfg(**kw):
        return C.byref(A.DelayConfig(**kw).to_c())

    assert est(f, f, None, 0, 8, 8, cfg(), None, i, None, None, None) == 0             # empty batch
    for D in (0, 128, 300, 1000, 16384, -256):
        assert est(f, f, None, 1, 8, 8, cfg(max_delay=D), None, i, None, None, None) == -1, D
    assert est(f, f, None, 1, 8, 8, cfg(margin=-1), None, i, None, None, None) == -1
    assert est(f, f, None, 1, 8, 8, cfg(min_peak=float("nan")), None, i, None, None, None) == -1
    assert est(f, f, None, 1, 8, 8, None, None, i, None, None, None) == -1
    assert est(f, f, None, -1, 8, 8, cfg(), None, i, None, None, None) == -1
    assert est(f, f, None, 1, 8, 4, cfg(), None, i, None, None, None) == -1              # stride < L
    assert est(None, f, None, 1, 8, 8, cfg(), None, i, None, None, None) == -1
    assert est(f, None, None, 1, 8, 8, cfg(), None, i, None, None, None) == -1
    assert est(f, f, None, 1, 8, 8, cfg(), i, None, f, None, None) == -1                 # shift is required
    al = lib.aec_delay_align
    g = np.zeros(64, dtype=np.float32).ctypes.data
    assert al(f, g, i, 0, 8, 8, 8, None) == 0
    assert al(f, g, i, -1, 8, 8, 8, None) == -1
    assert al(f, g, i, 1, 8, 4, 8, None) == -1
    assert al(f, g, i, 1, 8, 8, 4, None) == -1
    assert al(None, g, i, 1, 8, 8, 8, None) == -1
    assert al(f, None, i, 1, 8, 8, 8, None) == -1
    assert al(f, g, None, 1, 8, 8, 8, None) == -1
    assert al(f, f, i, 1, 8, 8, 8, None) == -1                                           # in place
    c1 = _lib.default_cfg(512)
    for fn in (lib.aec_stage1_run_host_ex, lib.aec_stage1_run_host_pcm16_ex):
        assert fn(None, f, f, g, None, None, None, 1, 8, 8, 8, C.byref(c1), cfg(), None, None) == -1


def _wav_set(tmp_path, n_utt=6, bulk_delay=700, subdirs=False):
    from scipy.io import wavfile

    wav = tmp_path / "wav"
    wav.mkdir()
    for i in range(n_utt):
        u = synth.make_utterance(i, 6000 + 100 * i, rir_len=512, bulk_delay=bulk_delay)
        for key, src in (("farend_speech", "far"), ("nearend_mic", "mic"), ("echo", "echo"), ("nearend_speech", "near")):
            d = wav / key if subdirs else wav
            d.mkdir(exist_ok=True)
            pcm = np.clip(np.rint(u[src] * 32768.0), -32768, 32767).astype(np.int16)
            wavfile.write(str(d / wav2h5.WAV_PATTERNS[key].format(idx=i)), 16000, pcm)
    return wav


def _fake_aligning_runner(far, mic, n):
    """stands in for Stage1Runner(align=...): (err, echo, shift) with a recognisable shift per row"""
    err = np.asarray(mic, np.float32) * np.float32(0.5) if mic.dtype != np.int16 else mic.astype(np.float32) / 65536
    return err, err * 2, (np.arange(far.shape[0], dtype=np.int32) * 7 + 3)


def _fake_runner(far, mic, n):
    return _fake_aligning_runner(far, mic, n)[:2]


def test_generators_write_the_far_shift_only_when_aligning(tmp_path):
    from acoustic_echo_cancellation_b200 import h5lite

    wav = _wav_set(tmp_path)
    files = {}
    for tag, runner in (("plain", _fake_runner), ("aligned", _fake_aligning_runner)):
        for native in (True, False):
            d = tmp_path / f"h5_{tag}_{native}"
            d.mkdir()
            args = types.SimpleNamespace(train_path=str(wav), h5_path=str(d), list_path=str(d), sr=16000)
            paths = wav2h5.create_h5_train(args, runner=runner, batch=4, h5=h5lite, native_writer=native)
            files[(tag, native)] = {os.path.basename(p): open(p, "rb").read() for p in paths}
            for j, p in enumerate(sorted(paths, key=lambda p: int(p.split("tr_")[-1][:-3]))):
                with h5lite.File(p, "r") as r:
                    names = set(r.keys())
                    if tag == "plain":
                        assert "stage1_far_shift" not in names
                    else:
                        sh = np.array(r["stage1_far_shift"])
                        assert sh.dtype == np.float32 and sh.shape == (1,)
                        assert len(names) == 7
    assert files[("plain", True)] == files[("plain", False)]
    assert files[("aligned", True)] == files[("aligned", False)]
    # test form: inside each numbered group
    d = tmp_path / "tt"
    d.mkdir()
    args = types.SimpleNamespace(val_path=str(wav), h5_path=str(d), list_path=str(d), sr=16000)
    path = wav2h5.create_h5_test(args, runner=_fake_aligning_runner, batch=4, h5=h5lite)
    with h5lite.File(path, "r") as r:
        shifts = sorted(float(np.array(r[g]["stage1_far_shift"])[0]) for g in r.keys())
    assert shifts == sorted([3.0, 10.0, 17.0, 24.0, 3.0, 10.0])


def test_val_form_writes_the_far_shift(tmp_path):
    from acoustic_echo_cancellation_b200 import h5lite

    wav = _wav_set(tmp_path, n_utt=3, subdirs=True)
    d = tmp_path / "h5"
    d.mkdir()
    args = types.SimpleNamespace(val_path=str(wav), h5_path=str(d), list_path=str(d), sr=16000)
    path = wav2h5.create_h5_val(args, runner=_fake_aligning_runner, batch=4, h5=h5lite)
    with h5lite.File(path, "r") as r:
        for g in r.keys():
            assert set(r[g].keys()) == {"mic", "ref", "near", "echo", "stage1_error", "stage1_echo", "stage1_far_shift"}


def test_align_flag_builds_an_aligning_runner():
    p = wav2h5.build_parser("train")
    assert wav2h5.runner_from_args(p.parse_args([])).align is None
    r = wav2h5.runner_from_args(p.parse_args(["--stage1_align_max_delay", "4096"]))
    assert r.align == A.DelayConfig(max_delay=4096)


# ------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------
def _torch():
    import torch

    return torch


def _cuda(a):
    return _torch().from_numpy(np.ascontiguousarray(a)).cuda()


def _est(far, mic, D, n=None, **kw):
    torch = _torch()
    r = A.estimate_delay(far, mic, A.DelayConfig(max_delay=D, **kw), n_samples=n, return_corr=True)
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in r]


def _rule(delay, peak, margin=128, min_peak=0.1):
    return np.where(peak >= np.float32(min_peak), np.maximum(delay - margin, 0), 0)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [256, 2048, 8192])
def test_estimate_matches_the_oracle_on_every_row(D):
    far, mic, n, names, ref, _ = _oracle(D)
    delay, shift, peak, corr = _est(_cuda(far), _cuda(mic), D, _cuda(n))
    err = np.abs(corr - ref["corr"]).max(axis=1)
    assert err.max() <= CORR_TOL, dict(zip(names, err))
    assert np.abs(peak - ref["peak"]).max() <= CORR_TOL
    a = np.sort(np.abs(ref["corr"]), axis=1)
    clear = (a[:, -1] - a[:, -2]) > 1e-3
    assert clear.sum() >= len(names) - 6
    assert np.array_equal(delay[clear], ref["delay"][clear]), [nm for nm, c, x, y in zip(names, clear, delay, ref["delay"])
                                                               if c and x != y]
    assert np.array_equal(shift, _rule(delay, peak))
    assert np.array_equal(shift[clear], ref["shift"][clear])
    for name in ("silent_far", "dc_only", "n0"):
        i = names.index(name)
        assert delay[i] == 0 and peak[i] == 0 and shift[i] == 0 and not corr[i].any(), name
    lv = [names.index(f"level{x:g}") for x in LEVELS]
    assert len(set(delay[lv])) == 1


@pytest.mark.gpu
def test_estimate_launch_shapes_invariance_and_canaries():
    torch = _torch()
    D = 2048
    far, mic, n, names, ref, _ = _oracle(D)
    B, L = far.shape
    base = _est(_cuda(far), _cuda(mic), D, _cuda(n))
    again = _est(_cuda(far), _cuda(mic), D, _cuda(n))
    assert all(np.array_equal(x, y) for x, y in zip(base, again))              # run to run
    for b in (0, 5, names.index("n1"), B - 1):                                  # every row as in a batch of one
        one = _est(_cuda(far[b:b + 1, :n[b]]), _cuda(mic[b:b + 1, :n[b]]), D)
        assert all(np.array_equal(x[0], y[b]) for x, y in zip(one, base)), b
    # rows 1 float off 16-byte alignment, odd stride, canaries beyond every output
    stride = L + 3
    buf = torch.zeros((2, B * stride + 1), device="cuda")
    for s, a in enumerate((far, mic)):
        buf[s, 1:1 + B * stride].view(B, stride)[:, :L] = _cuda(a)
    lib = _lib.load()
    c = A.DelayConfig(max_delay=D).to_c()
    canary = -777
    dl = torch.full((B + 4,), canary, dtype=torch.int32, device="cuda")
    sh = dl.clone()
    pk = torch.full((B + 4,), float(canary), device="cuda")
    co = torch.full((B * (D + 1) + 16,), float(canary), device="cuda")
    nd = _cuda(n)
    rc = lib.aec_delay_estimate(buf[0, 1:].data_ptr(), buf[1, 1:].data_ptr(), nd.data_ptr(), B, L, stride, C.byref(c),
                                dl.data_ptr(), sh.data_ptr(), pk.data_ptr(), co.data_ptr(), None)
    _lib.check(rc, "aec_delay_estimate")
    torch.cuda.synchronize()
    got = [dl[:B].cpu().numpy(), sh[:B].cpu().numpy(), pk[:B].cpu().numpy(), co[:B * (D + 1)].view(B, D + 1).cpu().numpy()]
    assert all(np.array_equal(x, y) for x, y in zip(got, base))
    assert (dl[B:] == canary).all() and (sh[B:] == canary).all() and (pk[B:] == canary).all()
    assert (co[B * (D + 1):] == canary).all()
    # nullable delay / peak / corr: same shift
    sh2 = torch.full((B,), canary, dtype=torch.int32, device="cuda")
    _lib.check(lib.aec_delay_estimate(buf[0, 1:].data_ptr(), buf[1, 1:].data_ptr(), nd.data_ptr(), B, L, stride,
                                      C.byref(c), None, sh2.data_ptr(), None, None, None), "aec_delay_estimate")
    assert np.array_equal(sh2.cpu().numpy(), base[1])


@pytest.mark.gpu
def test_estimate_batch_sizes():
    torch = _torch()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    D = 256
    for B, L in ((1, 3000), (sms + 1, 3000), (65538, 300)):
        rng = np.random.default_rng(B)
        far = rng.standard_normal((B, L)).astype(np.float32)
        mic = np.zeros_like(far)
        d = rng.integers(0, 100, B)
        for b in range(B):
            mic[b, d[b]:] = far[b, :L - d[b]]
        mic += 0.1 * rng.standard_normal((B, L)).astype(np.float32)
        delay, shift, peak, corr = _est(_cuda(far), _cuda(mic), D, margin=16)
        assert np.array_equal(delay, d), B
        for b in sorted({0, B // 2, B - 1}):
            one = _est(_cuda(far[b:b + 1]), _cuda(mic[b:b + 1]), D, margin=16)
            assert all(np.array_equal(x[0], y[b]) for x, y in zip(one, (delay, shift, peak, corr))), (B, b)
        if B < 1000:
            ref = DO.estimate(far, mic, DO.DelayConfig(max_delay=D, margin=16))
            assert np.abs(corr - ref["corr"]).max() <= CORR_TOL


@pytest.mark.gpu
def test_align_is_a_bit_exact_shift():
    torch = _torch()
    B, L = 6, 5000
    n = np.array([5000, 4000, 3000, 5000, 5000, 5000])
    far = torch.randn(B, L, device="cuda")
    shift_np = np.array([0, 1, 4000, L, L + 9, -5], dtype=np.int32)             # 0, 1, n_b, L, > L, negative = 0
    out = torch.full((B, L + 7), -5.0, device="cuda")
    A.align_far(far, _cuda(shift_np), out=out[:, :L])
    ref = torch.zeros(B, L, device="cuda")
    for b, s in enumerate(shift_np):
        s = max(int(s), 0)
        if s < L:
            ref[b, s:] = far[b, :L - s]
    assert torch.equal(out[:, :L], ref)
    assert (out[:, L:] == -5.0).all()
    # unaligned, odd-stride input
    buf = torch.zeros(B * (L + 1) + 1, device="cuda")
    v = buf[1:].view(B, L + 1)[:, :L]
    v.copy_(far)
    assert torch.equal(A.align_far(v, _cuda(shift_np)), ref)
    assert np.array_equal(DO.align(far.cpu().numpy(), shift_np), ref.cpu().numpy())
    del n


@pytest.mark.gpu
@pytest.mark.parametrize("frame,algo", [(512, 0), (512, 1), (512, 2), (512, 3), (1024, 0), (1024, 2)])
def test_stage1_align_equals_align_then_stage1(frame, algo):
    torch = _torch()
    d = synth.make_batch(0, 4, 30000, rir_len=512, bulk_delay=1500)
    far, mic = _cuda(d["far"]), _cuda(d["mic"])
    n = _cuda(np.array([30000, 20000, 9000, 1]))
    cfg = A.Stage1Config(frame=frame, partitions=4, algo=algo)
    dc = A.DelayConfig(max_delay=4096)
    err, erle, shift = A.stage1_aec(far, mic, cfg, n_samples=n, return_erle=True, align=dc, return_shift=True)
    _, sh, _ = A.estimate_delay(far, mic, dc, n_samples=n)
    ref, ref_erle = A.stage1_aec(A.align_far(far, sh), mic, cfg, n_samples=n, return_erle=True)
    torch.cuda.synchronize()
    assert torch.equal(shift, sh) and torch.equal(err, ref) and torch.equal(erle, ref_erle)
    assert int(shift[0]) > 1000


@pytest.mark.gpu
@pytest.mark.parametrize("algo", [2, 3])
def test_alignment_restores_erle_on_a_200ms_delay(algo):
    """6 s, 200 ms bulk delay, P = 4.  The NLMS step (algo 2) is back at the noise floor; the Kalman step (algo 3)
    converges more slowly and reaches 35 dB over the second half only without any delay (float64 oracle: 34.9 dB
    undelayed, 33.0 dB aligned -- the 128-sample margin plus the response's onset leave 1024 - 131 taps for the 1024-tap
    response), so it is held to within 2.5 dB of the undelayed utterance through the same kernel"""
    u = synth.make_utterance(0, 96000, bulk_delay=3200)
    u0 = synth.make_utterance(0, 96000)
    far, mic = _cuda(u["far"][None]), _cuda(u["mic"][None])
    cfg = A.Stage1Config(partitions=4, algo=algo)
    plain = A.stage1_aec(far, mic, cfg).cpu().numpy()[0]
    aligned = A.stage1_aec(far, mic, cfg, align=A.DelayConfig()).cpu().numpy()[0]
    undelayed = A.stage1_aec(_cuda(u0["far"][None]), _cuda(u0["mic"][None]), cfg).cpu().numpy()[0]
    m = (96000 // 256) * 256
    assert _erle_second_half(u["mic"], plain[:m]) < 3.0
    erle = _erle_second_half(u["mic"], aligned[:m])
    if algo == A.ALGO_PBFDAF:
        assert erle >= 35.0
    else:
        assert erle >= 30.0 and erle >= _erle_second_half(u0["mic"], undelayed[:m]) - 2.5


@pytest.mark.gpu
@pytest.mark.parametrize("pcm16", [False, True])
def test_host_pipeline_align_equals_the_device_path(pcm16):
    torch = _torch()
    B, L = 40, 12000
    d = synth.make_batch(10, B, L, rir_len=512, bulk_delay=900)
    n = np.random.default_rng(1).integers(0, L + 1, B).astype(np.int64)
    n[0] = L
    if pcm16:
        far_h = np.clip(np.rint(d["far"] * 32768), -32768, 32767).astype(np.int16)
        mic_h = np.clip(np.rint(d["mic"] * 32768), -32768, 32767).astype(np.int16)
        far_f, mic_f = far_h.astype(np.float32) / 32768, mic_h.astype(np.float32) / 32768
    else:
        far_h, mic_h, far_f, mic_f = d["far"], d["mic"], d["far"], d["mic"]
    cfg = A.Stage1Config(partitions=4, algo=A.ALGO_PBFDAF)
    dc = A.DelayConfig(max_delay=2048)
    err_d, erle_d, shift_d = A.stage1_aec(_cuda(far_f), _cuda(mic_f), cfg, n_samples=_cuda(n), return_erle=True,
                                          align=dc, return_shift=True)
    _, _, peak_d = A.estimate_delay(_cuda(far_f), _cuda(mic_f), dc, n_samples=_cuda(n))
    torch.cuda.synchronize()
    pipe = A.HostPipeline(16, L, slots=2)
    try:
        outs = []
        for deferred in (False, True):
            err = np.zeros((B, L), np.float32)
            erle = np.zeros(B, np.float32)
            shift = np.zeros(B, np.int32)
            peak = np.zeros(B, np.float32)
            pipe.run(far_h, mic_h, cfg, n_samples=n, err=err, erle=erle, align=dc, shift=shift, peak=peak,
                     wait=not deferred)
            if deferred:
                pipe.wait()
            outs.append((err, erle, shift, peak))
        for err, erle, shift, peak in outs:
            assert np.array_equal(err, err_d.cpu().numpy())
            assert np.array_equal(erle, erle_d.cpu().numpy())
            assert np.array_equal(shift, shift_d.cpu().numpy())
            assert np.array_equal(peak, peak_d.cpu().numpy())
        assert (outs[0][2] > 0).sum() >= B // 2
        # launches: align=None is the stage-1 call alone (+ the two PCM16 conversions per slice)
        small = slice(0, 8)
        per_slice = 3 if pcm16 else 1
        A.launch_count(reset=True)
        pipe.run(far_h[small], mic_h[small], cfg, n_samples=n[small])
        assert A.launch_count() == per_slice
        A.launch_count(reset=True)
        pipe.run(far_h[small], mic_h[small], cfg, n_samples=n[small], align=dc)
        assert A.launch_count() == per_slice + 2
        with pytest.raises(ValueError):
            pipe.run(far_h, mic_h, cfg, shift=np.zeros(B, np.int32))
    finally:
        pipe.close()


@pytest.mark.gpu
def test_create_h5_train_with_the_align_flag(tmp_path):
    from acoustic_echo_cancellation_b200 import h5lite

    torch = _torch()
    wav = _wav_set(tmp_path, n_utt=9, bulk_delay=1200)
    d = tmp_path / "h5"
    d.mkdir()
    a = wav2h5.build_parser("train").parse_args(["--train_path", str(wav), "--h5_path", str(d), "--list_path", str(d),
                                                 "--stage1_algo", "ols-nlms", "--stage1_align_max_delay", "2048"])
    paths = wav2h5.create_h5(a, runner=wav2h5.runner_from_args(a), batch=4, h5=h5lite)
    cfg = A.Stage1Config(algo=A.ALGO_PBFDAF, partitions=4)
    dc = A.DelayConfig(max_delay=2048)
    for p in paths:
        with h5lite.File(p, "r") as r:
            far = np.array(r["farend_speech"])
            mic = np.array(r["nearend_mic"])
            err, shift = A.stage1_aec(_cuda(far[None]), _cuda(mic[None]), cfg, align=dc, return_shift=True)
            torch.cuda.synchronize()
            assert np.array_equal(np.array(r["stage1_far_shift"]), np.array([shift.item()], np.float32))
            assert np.array_equal(np.array(r["stage1_error"]), err.cpu().numpy()[0])
            assert shift.item() > 1000
