"""Streaming Stage 2 (aec_stage2_run_stream, Stage2Stream, AecStream): Little_net with its GRU state, last input hop and
pending overlap-add half-frame carried from one call to the next.

CPU: the stateful float64 oracle in ragged chunks equals ``stage2_little_net(in_norm=False)`` on the whole signal; the
state size follows the documented layout; every refusal and argument error returns its code without a GPU and without a
launch.
GPU (-m gpu): chunked calls equal one call bit for bit (ragged per-row schedules, 0-, 1-, 16- and 625-hop calls, aligned
and unaligned rows, batch sizes on both sides of the kernel's persistent-grid threshold); one call and a flush against
the float64 oracle and, to 1e-6 relative, against ``LittleNetInference(in_norm=False)``; the same over 10 s utterances in
160-sample chunks, with the state after 625 hops; the stored state against the oracle state and a warm start from it;
``Stage2Stream`` chunking, flush and reset; hygiene; ``AecStream`` end to end and through flushes and resets of some
rows; the kernel the profiler names.
"""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import aec_oracle as O
from oracle.stage2_oracle_stream import little_net_stream

from acoustic_echo_cancellation_b200 import _lib

H = 256
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
TOL_NET = 2e-4       # x max|ref| per row, the bar of test_stage2_kernels
STATE_BYTES = 16 + 4 * 32 + 3 * 4 * H       # frames (+ reserved), h, mic_prev, ref_prev, ola


def _weights():
    g = np.load(os.path.join(GOLDEN, "reference_stage2.npz"))
    return {k[2:]: g[k] for k in g.files if k.startswith("w_")}, g["erb"]


def _oracle_chunked(mic, ref, erb, w, chunks):
    """the oracle fed sample chunks as a caller would: whole hops go in, the rest waits; then one zero-padded hop"""
    pend_m, pend_r, outs, st = np.zeros(0), np.zeros(0), [], None
    pos = 0
    for n in chunks:
        pend_m = np.concatenate([pend_m, mic[pos:pos + n]])
        pend_r = np.concatenate([pend_r, ref[pos:pos + n]])
        pos += n
        c = len(pend_m) // H * H
        o, st = little_net_stream(pend_m[:c], pend_r[:c], erb, w, st)
        outs.append(o)
        pend_m, pend_r = pend_m[c:], pend_r[c:]
    assert pos == len(mic)
    last_m, last_r = np.zeros(H), np.zeros(H)
    last_m[:len(pend_m)], last_r[:len(pend_r)] = pend_m, pend_r
    o, st = little_net_stream(last_m, last_r, erb, w, st)
    outs.append(o)
    return np.concatenate(outs), st


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("L", (1, 255, 256, 257, 511, 512, 513, 16 * H, 12365))
def test_oracle_stream_in_chunks_equals_the_whole_signal(L):
    w, erb = _weights()
    rng = np.random.default_rng(L)
    mic, ref = 0.1 * rng.standard_normal(L), 0.2 * rng.standard_normal(L)
    want = O.stage2_little_net(mic[None], ref[None], erb, w, in_norm=False)[0]
    for _ in range(3):
        chunks, pos = [], 0
        while pos < L:
            n = min(int(rng.choice([0, 1, 255, 256, 257, 160, 3 * H + 7])), L - pos)
            chunks.append(n)
            pos += n
        got, st = _oracle_chunked(mic, ref, erb, w, chunks)
        assert got.shape == want.shape
        assert st["frames"] == L // H + 1
        if want.size:
            assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_state_bytes_follow_the_layout():
    assert STATE_BYTES == 3216
    assert _lib.load().aec_stage2_state_bytes() == STATE_BYTES


def test_refusals_and_argument_errors_need_no_gpu():
    import acoustic_echo_cancellation_b200 as A
    lib = _lib.load()
    nb = STATE_BYTES
    st = np.zeros(2 * nb + 64, dtype=np.uint8)
    s16 = (st.ctypes.data + 15) // 16 * 16
    buf = np.zeros(8192, dtype=np.float32)
    f = buf.ctypes.data
    arrs = [np.zeros(96 * 64, dtype=np.float32) for _ in range(8)]
    good = _lib.Stage2Weights(*[a.ctypes.data for a in arrs])
    null_field = _lib.Stage2Weights(*[a.ctypes.data for a in arrs[:7]], None)
    misaligned = _lib.Stage2Weights(arrs[0].ctypes.data + 2, *[a.ctypes.data for a in arrs[1:]])
    run = lib.aec_stage2_run_stream
    g = C.byref(good)
    A.launch_count(reset=True)
    for bands in (31, 16, 64, 0):
        assert run(f, f, f, g, f, None, 1, 256, 256, 256, s16, nb, bands, None) == -2
    assert run(f, f, f, g, f, None, 1, 256, 256, 256, None, nb, 32, None) == -1                # null state
    assert run(f, f, f, g, f, None, 1, 256, 256, 256, s16 + 4, nb, 32, None) == -1             # misaligned state
    assert run(f, f, f, g, f, None, 1, 256, 256, 256, s16, nb - 16, 32, None) == -1            # stride < bytes
    assert run(f, f, f, g, f, None, 1, 256, 256, 256, s16, nb + 8, 32, None) == -1             # stride % 16
    assert run(f, f, f, None, f, None, 1, 256, 256, 256, s16, nb, 32, None) == -1              # no weights
    assert run(f, f, f, C.byref(null_field), f, None, 1, 256, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f, C.byref(misaligned), f, None, 1, 256, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f, g, f, None, -1, 256, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f, g, f, None, 1, -1, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f, g, f, None, 1, 256, 128, 256, s16, nb, 32, None) == -1                 # in_stride < L
    assert run(f, f, f, g, f, None, 1, 256, 256, 128, s16, nb, 32, None) == -1                 # out_stride < L
    assert run(None, f, f, g, f, None, 1, 256, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f + 2, g, f, None, 1, 256, 256, 256, s16, nb, 32, None) == -1             # misaligned bank
    assert run(f, f, f, g, None, None, 1, 256, 256, 256, s16, nb, 32, None) == -1
    assert run(f, f, f, g, f, None, 0, 256, 256, 256, s16, nb, 32, None) == 0                  # empty batch
    assert run(f, f, f, g, f, None, 3, 0, 0, 0, s16, nb, 32, None) == 0                        # empty chunk
    init = lib.aec_stage2_state_init
    assert init(None, 1, nb, None, None) == -1
    assert init(s16 + 8, 1, nb, None, None) == -1
    assert init(s16, 1, nb - 16, None, None) == -1
    assert init(s16, 1, nb + 4, None, None) == -1
    assert init(s16, -1, nb, None, None) == -1
    assert init(s16, 0, nb, None, None) == 0
    assert A.launch_count() == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _sms():
    torch = _torch()
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _signals(B, L, seed):
    """mic / ref [B, L] float32 on the device, a different level per row (a row read in another's place shows)"""
    torch = _torch()
    g = torch.Generator(device="cuda").manual_seed(seed)
    gain = 0.1 + 0.2 * torch.rand(B, 1, device="cuda", generator=g)
    return (gain * torch.randn(B, L, device="cuda", generator=g),
            gain.flip(0) * torch.randn(B, L, device="cuda", generator=g))


def _stream(B):
    import acoustic_echo_cancellation_b200 as A
    w, erb = _weights()
    return A.Stage2Stream(B, w, erb)


class _Raw:
    """Direct aec_stage2_run_stream calls on B streams (the C ABI, without Stage2Stream's pending samples)."""

    def __init__(self, B):
        self.torch = _torch()
        self.s = _stream(B)
        self.lib = _lib.load()

    def call(self, mic, ref, ns, unaligned=False):
        """mic, ref: [B, L] device tensors; ns: int64 [B] device tensor or list (the kernel consumes ns // 256 hops).
        Returns out [B, L] (device) after checking the canaries past L."""
        torch = self.torch
        B, L = mic.shape
        stride = L + 1 if unaligned else (L + 3) // 4 * 4
        off = 1 if unaligned else 0
        buf = torch.zeros((2, B * stride + 8), dtype=torch.float32, device="cuda")
        for i, x in enumerate((mic, ref)):
            buf[i, off:off + B * stride].view(B, stride)[:, :L] = x
        out = torch.full((B, stride + 4), 7.0, device="cuda")
        n_t = torch.as_tensor(ns, dtype=torch.int64, device="cuda")
        rc = self.lib.aec_stage2_run_stream(buf[0, off:].data_ptr(), buf[1, off:].data_ptr(), self.s.erb.data_ptr(),
                                            C.byref(self.s._cw), out.data_ptr(), n_t.data_ptr(), B, L, stride,
                                            stride + 4, self.s.state.data_ptr(), self.s.state_stride, 32,
                                            int(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc, "aec_stage2_run_stream")
        assert bool((out[:, L:] == 7.0).all()), "written past L"
        return out[:, :L]


def _schedules(B, nhops, rng, long_row=None):
    """per stream, sample counts per call: 0-, 1- and 16-hop calls with a tail the caller keeps; row 0 alternates 0 and
    1 hop; ``long_row`` takes all its hops in one call"""
    out = []
    for b in range(B):
        sched, done = [], 0
        while done < nhops:
            if b == long_row:
                k = nhops
            elif b == 0:
                k = 1 if len(sched) % 3 else 0
            else:
                k = int(rng.choice([0, 1, 1, 2, 16]))
            k = min(k, nhops - done)
            sched.append(k * H + int(rng.integers(0, H)))
            done += k
        out.append(sched)
    return out


def _chunked(raw, mic, ref, scheds, unaligned=False):
    """run the schedules; returns the concatenated output of each row [B, sum of blocks] (device) and its length"""
    torch = _torch()
    B, N = mic.shape
    pos = torch.zeros(B, dtype=torch.int64, device="cuda")
    got = torch.zeros((B, N), device="cuda")
    acc = torch.zeros(B, dtype=torch.int64, device="cuda")
    first = torch.ones(B, dtype=torch.bool, device="cuda")
    for k in range(max(len(s) for s in scheds)):
        ns = torch.tensor([s[k] if k < len(s) else 0 for s in scheds], dtype=torch.int64, device="cuda")
        Lc = max(int(ns.max()), 1)
        j = torch.arange(Lc, device="cuda")[None, :]
        idx = (pos[:, None] + j).clamp(max=N - 1)
        valid = (j < ns[:, None]) & (pos[:, None] + j < N)
        mk = torch.where(valid, torch.gather(mic, 1, idx), 0.0)
        rk = torch.where(valid, torch.gather(ref, 1, idx), 0.0)
        out = raw.call(mk, rk, ns, unaligned=unaligned)
        hops = ns // H
        n_out = (hops - (first & (hops > 0)).to(torch.int64)) * H
        first &= hops == 0
        assert not bool(torch.where(j < n_out[:, None], 0.0, out).any()), "non-zero past the row's blocks"
        dst = (acc[:, None] + j).clamp(max=N - 1)
        got.scatter_(1, dst, torch.where(j < n_out[:, None], out, torch.gather(got, 1, dst)))
        acc += n_out
        pos += hops * H
    return got, acc


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
# B: one partial CTA; the largest batch with one stream per warp (8 x SM count); batches whose warps walk several streams
@pytest.mark.gpu
@pytest.mark.parametrize("Bspec", ("3", "8sms", "8sms+5", "24sms+2"))
def test_chunked_equals_one_call_bit_for_bit(Bspec):
    torch = _torch()
    B = 3 if Bspec == "3" else int(Bspec.split("sms")[0]) * _sms() + int(Bspec.split("sms")[1] or 0)
    nhops = 40
    mic, ref = _signals(B, nhops * H, B)
    scheds = _schedules(B, nhops, np.random.default_rng(B), long_row=1)
    raw = _Raw(B)
    got, acc = _chunked(raw, mic, ref, scheds)
    one = _Raw(B).call(mic, ref, [nhops * H] * B)
    assert bool((acc == (nhops - 1) * H).all())
    assert torch.equal(got[:, :(nhops - 1) * H], one[:, :(nhops - 1) * H])
    assert raw.s.state_views()["frames"].cpu().tolist() == [nhops] * B


@pytest.mark.gpu
def test_chunked_equals_one_call_with_a_625_hop_call_and_unaligned_rows():
    torch = _torch()
    B, nhops = 5, 640
    mic, ref = _signals(B, nhops * H, 17)
    scheds = _schedules(B, nhops, np.random.default_rng(5), long_row=2)
    scheds[3] = [625 * H + 11, 15 * H]
    for unaligned in (False, True):
        got, acc = _chunked(_Raw(B), mic, ref, scheds, unaligned=unaligned)
        one = _Raw(B).call(mic, ref, [nhops * H] * B, unaligned=not unaligned)
        assert bool((acc == (nhops - 1) * H).all())
        assert torch.equal(got[:, :(nhops - 1) * H], one[:, :(nhops - 1) * H])


LENGTHS = (1, 255, 256, 257, 511, 512, 513, 16 * H, 12365)


def _one_call_and_flush(mic, ref, lengths):
    """Stage2Stream: one process call (row b: its first lengths[b] samples) and a flush; per-row outputs (numpy)"""
    torch = _torch()
    s = _stream(mic.shape[0])
    n = torch.as_tensor(lengths, dtype=torch.int64, device="cuda")
    o1, c1 = s.process(mic, ref, n)
    o2, c2 = s.flush()
    o1, c1, o2, c2 = o1.cpu().numpy(), c1.cpu().numpy(), o2.cpu().numpy(), c2.cpu().numpy()
    return [np.concatenate([o1[b, :c1[b]], o2[b, :c2[b]]]) for b in range(mic.shape[0])]


@pytest.mark.gpu
def test_one_call_and_flush_against_the_float64_oracle():
    w, erb = _weights()
    mic, ref = _signals(len(LENGTHS), max(LENGTHS), 3)
    got = _one_call_and_flush(mic, ref, LENGTHS)
    m, r = mic.cpu().numpy().astype(np.float64), ref.cpu().numpy().astype(np.float64)
    for b, L in enumerate(LENGTHS):
        want = O.stage2_little_net(m[b:b + 1, :L], r[b:b + 1, :L], erb, w, in_norm=False)[0]
        assert got[b].shape == want.shape == ((L // H) * H,)
        if want.size:
            err = np.abs(got[b] - want).max() / np.abs(want).max()
            assert err <= TOL_NET, f"L={L}: {err:.3g}"


@pytest.mark.gpu
def test_one_call_and_flush_match_little_net_inference():
    """each frame goes through the one-shot kernels' operations in their order, but the two units are compiled
    separately and their outputs are not always bit-identical (up to ~4e-7 relative in a few samples were seen on a
    B200); the bar here is 1e-6 x max|LittleNetInference|, 200x tighter than the oracle bar"""
    import acoustic_echo_cancellation_b200 as A
    w, erb = _weights()
    net = A.LittleNetInference(w, erb)
    mic, ref = _signals(2 * len(LENGTHS), max(LENGTHS), 4)
    got = _one_call_and_flush(mic, ref, [L for L in LENGTHS for _ in range(2)])
    for i, L in enumerate(LENGTHS):
        want = net(mic[2 * i:2 * i + 2, :L].contiguous(), ref[2 * i:2 * i + 2, :L].contiguous(), in_norm=False)
        want = want.cpu().numpy()
        for r in range(2):
            assert got[2 * i + r].shape == want[r].shape
            if want[r].size:
                err = np.abs(got[2 * i + r] - want[r]).max() / np.abs(want[r]).max()
                assert err <= 1e-6, f"L={L} row {r}: {err:.3g}"


@pytest.mark.gpu
def test_state_against_the_oracle_and_a_warm_start():
    torch = _torch()
    w, erb = _weights()
    B, k, n = 2, 37, 60
    mic, ref = _signals(B, n * H, 8)
    m64, r64 = mic.cpu().numpy().astype(np.float64), ref.cpu().numpy().astype(np.float64)
    raw = _Raw(B)
    raw.call(mic[:, :k * H].contiguous(), ref[:, :k * H].contiguous(), [k * H] * B)
    v = {name: t.cpu().numpy() for name, t in raw.s.state_views().items()}
    warm = _Raw(B)
    wv = warm.s.state_views()
    refs = []
    for b in range(B):
        _, st = little_net_stream(m64[b, :k * H], r64[b, :k * H], erb, w)
        assert v["frames"][b] == k
        assert np.array_equal(v["mic_prev"][b], mic[b, (k - 1) * H:k * H].cpu().numpy())
        assert np.array_equal(v["ref_prev"][b], ref[b, (k - 1) * H:k * H].cpu().numpy())
        assert np.abs(v["h"][b] - st["h"]).max() <= TOL_NET         # |h| < 1
        assert np.abs(v["ola"][b] - st["ola"]).max() <= TOL_NET * np.abs(st["ola"]).max()
        # warm start: the oracle's state, cast to float32, continued by the kernel
        wv["frames"][b] = k
        for name in ("h", "mic_prev", "ref_prev", "ola"):
            wv[name][b] = torch.as_tensor(st[name].astype(np.float32), device="cuda")
        want, _ = little_net_stream(m64[b, k * H:], r64[b, k * H:], erb, w, st)
        refs.append(want)
    out = warm.call(mic[:, k * H:].contiguous(), ref[:, k * H:].contiguous(), [(n - k) * H] * B).cpu().numpy()
    for b in range(B):
        assert refs[b].shape == ((n - k) * H,)
        assert np.abs(out[b] - refs[b]).max() <= TOL_NET * np.abs(refs[b]).max()


@pytest.mark.gpu
def test_whole_utterances_in_160_sample_chunks():
    """10 s rows (625 hops) at per-row gains, fed to Stage2Stream in 160-sample chunks and flushed: the carried GRU state
    and overlap-add must not drift from the one-shot path over a real utterance (the other comparisons with
    LittleNetInference and the oracle stop at 48 hops; the 640-hop test compares the streaming kernel with itself).
    Output within 1e-6 x max|LittleNetInference(in_norm=False)| (up to 6.0e-7 measured on these rows on a B200, of the
    same size at hop 48 as at hop 624: float32 rounding, not a drift) and TOL_NET of the float64 oracle;
    h and ola after 625 hops against little_net_stream's float64 state, as at 37 hops in
    test_state_against_the_oracle_and_a_warm_start."""
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    w, erb = _weights()
    B, n, chunk = 4, 625 * H, 160
    mic, ref = _signals(B, n, 21)
    s = _stream(B)
    outs = []
    for pos in range(0, n, chunk):
        o, c = s.process(mic[:, pos:pos + chunk], ref[:, pos:pos + chunk])
        c = c.cpu().tolist()
        assert c == [c[0]] * B
        outs.append(o[:, :c[0]])
    v = {name: t.cpu().numpy() for name, t in s.state_views().items()}
    o, c = s.flush()
    assert c.cpu().tolist() == [H] * B
    got = torch.cat(outs + [o[:, :H]], dim=1).cpu().numpy()
    assert got.shape == (B, n)
    want = A.LittleNetInference(w, erb)(mic, ref, in_norm=False).cpu().numpy()
    m64, r64 = mic.cpu().numpy().astype(np.float64), ref.cpu().numpy().astype(np.float64)
    want64 = O.stage2_little_net(m64, r64, erb, w, in_norm=False)
    for b in range(B):
        err = np.abs(got[b] - want[b]).max() / np.abs(want[b]).max()
        assert err <= 1e-6, f"row {b}: {err:.3g} x max|LittleNetInference|"
        err = np.abs(got[b] - want64[b]).max() / np.abs(want64[b]).max()
        assert err <= TOL_NET, f"row {b}: {err:.3g} x max|oracle|"
        _, st = little_net_stream(m64[b], r64[b], erb, w)
        assert v["frames"][b] == 625
        assert np.abs(v["h"][b] - st["h"]).max() <= TOL_NET         # |h| < 1
        assert np.abs(v["ola"][b] - st["ola"]).max() <= TOL_NET * np.abs(st["ola"]).max()


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", (1, 160, 333))
def test_stage2_stream_any_chunk_length(chunk):
    torch = _torch()
    B, n = 3, (6 if chunk == 1 else 40) * H + 77
    mic, ref = _signals(B, n, 40 + chunk)
    s = _stream(B)
    outs = [[] for _ in range(B)]
    for pos in range(0, n, chunk):
        o, c = s.process(mic[:, pos:pos + chunk], ref[:, pos:pos + chunk])
        c = c.cpu().tolist()
        assert not bool(o[:, max(c):].any())
        for r in range(B):
            outs[r].append(o[r, :c[r]])
    o, c = s.flush()
    for r in range(B):
        outs[r].append(o[r, :int(c[r])])
    want = _one_call_and_flush(mic, ref, [n] * B)
    for r in range(B):
        got = torch.cat(outs[r]).cpu().numpy()
        assert got.shape == ((n // H) * H,)
        assert np.array_equal(got, want[r])


@pytest.mark.gpu
def test_stage2_stream_flush_and_reset_of_some_rows():
    torch = _torch()
    B, n, cut = 4, 30 * H + 50, 11 * H + 100
    mic, ref = _signals(B, n, 9)
    s = _stream(B)
    o1, c1 = s.process(mic[:, :cut], ref[:, :cut])
    of, cf = s.flush([1])                 # row 1 ends at cut and restarts
    s.reset([3])                          # row 3 drops its state and pending samples, restarts at cut
    o2, c2 = s.process(mic[:, cut:], ref[:, cut:])
    o3, c3 = s.flush()
    assert int(cf[0]) == int(cf[2]) == int(cf[3]) == 0
    whole = _one_call_and_flush(mic, ref, [n] * B)
    head = _one_call_and_flush(mic[:, :cut].contiguous(), ref[:, :cut].contiguous(), [cut] * B)
    tail = _one_call_and_flush(mic[:, cut:].contiguous(), ref[:, cut:].contiguous(), [n - cut] * B)

    def seg(o, c, r):
        return o[r, :int(c[r])].cpu().numpy()

    for r in range(B):
        if r == 1:
            assert np.array_equal(np.concatenate([seg(o1, c1, r), seg(of, cf, r)]), head[r])
            assert np.array_equal(np.concatenate([seg(o2, c2, r), seg(o3, c3, r)]), tail[r])
        elif r == 3:
            assert np.array_equal(np.concatenate([seg(o2, c2, r), seg(o3, c3, r)]), tail[r])
        else:
            assert np.array_equal(np.concatenate([seg(o1, c1, r), seg(o2, c2, r), seg(o3, c3, r)]), whole[r])


@pytest.mark.gpu
def test_batch_and_call_hygiene():
    torch = _torch()
    mic, ref = _signals(3, 9 * H, 10)
    # run-to-run determinism and batch invariance (a row alone equals the same row in a batch)
    runs = []
    for _ in range(2):
        raw = _Raw(3)
        runs.append([raw.call(mic, ref, [9 * H, 5 * H + 3, 7 * H]), raw.call(mic, ref, [2 * H, 4 * H, 0])])
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    alone = _Raw(1)
    assert torch.equal(alone.call(mic[1:2], ref[1:2], [5 * H + 3])[0], runs[0][0][1])
    # a row without a whole hop leaves its state bytes untouched; canaries past state_bytes stay
    raw = _Raw(2)
    raw.call(mic[:2], ref[:2], [3 * H, 2 * H])
    big = _Raw(2)
    stride = big.s.state_stride + 64
    st = torch.full((2, stride), 0xA5, dtype=torch.uint8, device="cuda")
    st[:, :STATE_BYTES] = raw.s.state[:, :STATE_BYTES]
    big.s.state, big.s.state_stride = st, stride
    before = st.clone()
    out = big.call(mic[:2], ref[:2], [255, 0])
    assert torch.equal(st, before) and not bool(out.any())
    big.call(mic[:2], ref[:2], [H, 0])
    assert torch.equal(st[1], before[1]) and not torch.equal(st[0], before[0])
    assert bool((st[:, STATE_BYTES:] == 0xA5).all())
    # state_init: masked-out rows and the bytes past state_bytes stay untouched
    lib = _lib.load()
    st.fill_(0xA5)
    mask = torch.tensor([0, 1], dtype=torch.uint8, device="cuda")
    assert lib.aec_stage2_state_init(st.data_ptr(), 2, stride, mask.data_ptr(),
                                     int(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    assert bool((st[0] == 0xA5).all())
    assert not bool(st[1, :STATE_BYTES].any()) and bool((st[1, STATE_BYTES:] == 0xA5).all())


def _echo_signals(B, n, seed):
    from acoustic_echo_cancellation_b200 import synth
    torch = _torch()
    d = synth.make_batch(seed, B, n, sample_rate=16000, rir_len=1024)
    return torch.from_numpy(d["far"].astype(np.float32)).cuda(), torch.from_numpy(d["mic"].astype(np.float32)).cuda()


@pytest.mark.gpu
def test_aec_stream_end_to_end():
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    w, erb = _weights()
    B, n = 3, 40 * H + 77
    far, mic = _echo_signals(B, n, 12)
    cfg = A.Stage1Config(partitions=4, algo=A.ALGO_PBFDAF)
    err = A.stage1_aec(far, mic, cfg)
    want = A.LittleNetInference(w, erb)(err, far, in_norm=False).cpu().numpy()
    m = (n // H) * H
    results = []
    for chunk in (160, 333, n):
        s = A.AecStream(B, cfg, w, erb)
        outs = [[] for _ in range(B)]
        for pos in range(0, n, chunk):
            o, c = s.process(far[:, pos:pos + chunk], mic[:, pos:pos + chunk])
            for r in range(B):
                outs[r].append(o[r, :int(c[r])].cpu().numpy())
        o, c = s.flush()
        for r in range(B):
            outs[r].append(o[r, :int(c[r])].cpu().numpy())
        results.append([np.concatenate(x) for x in outs])
    for r in range(B):
        assert results[-1][r].shape == (m,) == want[r].shape
        err_r = np.abs(results[-1][r] - want[r]).max() / np.abs(want[r]).max()
        assert err_r <= TOL_NET, err_r
        for other in results[:-1]:
            assert np.array_equal(other[r], results[-1][r]), "chunked differs from unchunked"


# One call sequence for all six streams: ("p", chunk length) is a process call, ("flush", rows) / ("reset", rows) end the
# listed rows' segments.  Row 4 is flushed after 161 samples (no whole hop); row 1 mid-stream with 160 far-end samples
# held back by stage 1, then continues; row 3 is reset by bool mask; row 5 is flushed twice in a row (238 samples held
# back); rows 0 and 2 run through to the final flush of every row.
LIFECYCLE = [("p", 0), ("p", 1), ("p", 160), ("flush", [4]), ("p", 255), ("p", 4096), ("flush", [1]), ("p", 257),
             ("reset", [False, False, False, True, False, False]), ("p", 333), ("p", 256), ("flush", [5]),
             ("flush", [5]), ("p", 160), ("p", 4096), ("p", 1), ("p", 0), ("flush", None)]


def _lifecycle(s, far, mic):
    """run LIFECYCLE on AecStream s; returns per row the list of its segments (first sample, end, flushed, output), and
    checks every call's n_out and, after every call, the bookkeeping between the stages: stage 2 holds no pending
    samples (AecStream.flush relies on it) and AecStream holds back as many far-end samples as stage 1 holds"""
    torch = _torch()
    B = far.shape[0]
    pos, start, outs, segs = 0, [0] * B, [[] for _ in range(B)], [[] for _ in range(B)]

    def emitted(k):             # output samples of a segment of k samples before its flush
        return max(k // H - 1, 0) * H

    for op, arg in LIFECYCLE:
        if op == "p":
            o, c = s.process(far[:, pos:pos + arg], mic[:, pos:pos + arg])
            want = [emitted(pos + arg - start[r]) - emitted(pos - start[r]) for r in range(B)]
            pos += arg
        elif op == "flush":
            o, c = s.flush(arg)
            rows = range(B) if arg is None else arg
            want = [(H if pos - start[r] >= H else 0) if r in rows else 0 for r in range(B)]
        else:
            s.reset(arg)
            rows, c = [r for r in range(B) if arg[r]], None
        if c is not None:
            assert c.cpu().tolist() == want, f"{op} {arg}: n_out {c.cpu().tolist()} != {want}"
            for r in range(B):
                outs[r].append(o[r, :want[r]].cpu().numpy())
        assert not bool(s.s2._npend.any()), f"after {op} {arg}: stage 2 holds samples between calls"
        assert torch.equal(s._nfar, s.s1._npend), f"after {op} {arg}: far-end samples held back != stage 1's pending"
        if op != "p":
            for r in rows:
                segs[r].append((start[r], pos, op == "flush", np.concatenate(outs[r])))
                start[r], outs[r] = pos, []
    assert all(not o for o in outs)
    return segs


@pytest.mark.gpu
@pytest.mark.parametrize("P,algo", [(16, 3), (4, 2)], ids=("P16-kalman", "P4-nlms"))
def test_aec_stream_lifecycle(P, algo):
    """AecStream's own bookkeeping (the far-end samples stage 1 holds back, flush and reset of some rows while the others
    continue, chunks of 0, 1, 160, 255, 256, 257, 333 and 4096 samples): a mistake there mispairs the error and far-end
    samples of one stream and leaves the others right.  Every segment of every row between lifecycle events equals a
    fresh AecStream over that segment in one call (and a flush, where the segment was flushed) bit for bit, and
    LittleNetInference(in_norm=False)(stage1_aec(far, mic), far) on the segment within TOL_NET (a reset segment: the
    samples it produced); a flushed segment yields (num_frames(len) - 1) * 256 samples."""
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    w, erb = _weights()
    net = A.LittleNetInference(w, erb)
    cfg = A.Stage1Config(partitions=P, algo=algo)
    n = sum(a for op, a in LIFECYCLE if op == "p")
    far, mic = _echo_signals(6, n, 30 + P)
    segs = _lifecycle(A.AecStream(6, cfg, w, erb), far, mic)
    assert [len(x) for x in segs] == [1, 2, 1, 2, 2, 3]
    for r in range(6):
        for a, b, flushed, got in segs[r]:
            f, m = far[r:r + 1, a:b], mic[r:r + 1, a:b]
            fresh = A.AecStream(1, cfg, w, erb)
            o, c = fresh.process(f, m)
            one = [o[0, :int(c[0])]]
            if flushed:
                o, c = fresh.flush()
                one.append(o[0, :int(c[0])])
                assert got.shape == ((A.num_frames(b - a) - 1) * H,)
            assert np.array_equal(got, torch.cat(one).cpu().numpy()), f"row {r}, samples {a}:{b}"
            if got.size:
                want = net(A.stage1_aec(f.contiguous(), m.contiguous(), cfg), f.contiguous(), in_norm=False)
                want = want[0].cpu().numpy()
                err = np.abs(got - want[:got.size]).max() / np.abs(want).max()
                assert err <= TOL_NET, f"row {r}, samples {a}:{b}: {err:.3g}"


@pytest.mark.gpu
def test_profiler_names_the_stream_kernel():
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    mic, ref = _signals(1, 4 * H, 13)
    raw = _Raw(1)
    raw.call(mic, ref, [4 * H])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        raw.call(mic, ref, [4 * H])
        torch.cuda.synchronize()
    assert any("stage2_stream_kernel" in e.name for e in prof.events())
