"""Streaming stage 1 (aec_stage1_run_stream, Stage1Stream): the frame-512 overlap-save filters with their state carried
from one call to the next.

CPU: the stateful float64 oracle in chunks equals ``pbfdaf_ols`` on the whole signal exactly, at default and
non-default filter parameters; the state size follows the documented layout; every refusal and argument error returns
its code without a GPU and without a launch; the streaming unit builds exactly the 20 expected kernels.
GPU (-m gpu): chunked runs equal one ``stage1_aec`` call bit for bit for every build (ragged schedules, 0- and 1-block
calls, every T0 residue mod P, aligned and unaligned rows), at non-default filter parameters too (with the float64
oracle and the state after init and reset), and at full occupancy; each call's ERLE against its documented span; the
stored state against the float64 oracle; a warm start from the oracle's state; ``Stage1Stream`` chunking, reset and
echo / ERLE outputs; batch and call hygiene; the kernel the profiler names.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import aec_oracle as O
from oracle.aec_oracle_stream import pbfdaf_ols_stream

from acoustic_echo_cancellation_b200 import _lib

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "acoustic_echo_cancellation_b200", "csrc")
PS = (1, 2, 4, 8, 16)
ALGOS = (2, 3)
H = 256
K = 257


def _a16(n):
    return (n + 15) // 16 * 16


def _layout_bytes(P, algo):
    n = 16 + 4 * H + 2 * _a16(8 * P * K) + _a16(4 * K)
    return n + (_a16(4 * P * K) if algo == 3 else 0)


def _signals(B, n, seed):
    from acoustic_echo_cancellation_b200 import synth
    d = synth.make_batch(seed, B, n, sample_rate=16000, rir_len=1024)
    return d["far"].astype(np.float32), d["mic"].astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
# Non-default filter parameters: the PARAMS sets of test_stage1_builds.py for the overlap-save steps.  Across the sets
# every field a step rule reads (mu, delta, pb_lambda; kalman_a, kalman_lambda, kalman_c0, kalman_eps) leaves its default.
PARAMS = {
    2: [dict(pb_lambda=0.0, mu=1.0, delta=0.05), dict(pb_lambda=0.95, mu=0.2, delta=1.0)],
    3: [dict(kalman_a=0.99, kalman_lambda=0.5, kalman_c0=0.05, kalman_eps=1e-4),
        dict(kalman_a=0.995, kalman_lambda=0.8, kalman_c0=3.0, kalman_eps=1e-6)],
}


@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("algo", ALGOS)
def test_oracle_stream_in_chunks_equals_the_whole_signal(P, algo):
    """at the default parameters and at each PARAMS set of the step"""
    far, mic = _signals(1, 40 * H + 100, 70 + P + algo)
    far, mic = far[0].astype(np.float64), mic[0].astype(np.float64)
    for params in [{}] + PARAMS[algo]:
        cfg = O.AecConfig(partitions=P, algo=algo, **params)
        e_ref, y_ref = O.pbfdaf_ols(far, mic, cfg)
        rng = np.random.default_rng(P * 10 + algo)
        for _ in range(3):
            pos, state, es, ys = 0, None, [], []
            while pos < len(far):
                n = int(rng.choice([0, 1, 2, 3, 5])) * H + int(rng.integers(0, H))
                e, y, state = pbfdaf_ols_stream(far[pos:pos + n], mic[pos:pos + n], cfg, state)
                es.append(e)
                ys.append(y)
                pos += len(e)
                if len(e) == 0 and n >= len(far) - pos:
                    break
            assert state["blocks"] == len(far) // H
            assert np.array_equal(np.concatenate(es), e_ref), params
            assert np.array_equal(np.concatenate(ys), y_ref), params


@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("algo", ALGOS)
def test_state_bytes_follow_the_layout(P, algo):
    cfg = _lib.default_cfg(512, partitions=P, algo=algo)
    assert _lib.load().aec_stage1_state_bytes(C.byref(cfg)) == _layout_bytes(P, algo)


def test_refusals_and_argument_errors_need_no_gpu():
    import acoustic_echo_cancellation_b200 as A
    lib = _lib.load()
    good = _lib.default_cfg(512, algo=2)
    nbytes = lib.aec_stage1_state_bytes(C.byref(good))
    st = np.zeros(2 * nbytes + 64, dtype=np.uint8)
    s16 = (st.ctypes.data + 15) // 16 * 16
    f = np.zeros(4096, dtype=np.float32).ctypes.data
    unsupported = [_lib.default_cfg(512, algo=0), _lib.default_cfg(512, algo=1), _lib.default_cfg(1024, algo=2),
                   _lib.default_cfg(512, algo=3, variant=2128), _lib.default_cfg(512, algo=2, partitions=3),
                   _lib.default_cfg(512, algo=2, partitions=32)]
    A.launch_count(reset=True)
    for cfg in unsupported:
        assert lib.aec_stage1_state_bytes(C.byref(cfg)) == -2
        assert lib.aec_stage1_state_init(s16, 1, nbytes, None, C.byref(cfg), None) == -2
        assert lib.aec_stage1_run_stream(f, f, f, None, None, None, 1, 256, 256, 256, C.byref(cfg), s16, nbytes,
                                         None) == -2
    for cfg in (_lib.default_cfg(512, algo=2, partitions=0), _lib.default_cfg(512, algo=7)):
        assert lib.aec_stage1_state_bytes(C.byref(cfg)) == -1
    assert lib.aec_stage1_state_bytes(None) == -1
    run = lib.aec_stage1_run_stream
    g = C.byref(good)
    assert run(f, f, f, None, None, None, 1, 256, 256, 256, g, None, nbytes, None) == -1                # null state
    assert run(f, f, f, None, None, None, 1, 256, 256, 256, g, s16, nbytes - 16, None) == -1            # stride < bytes
    assert run(f, f, f, None, None, None, 1, 256, 256, 256, g, s16, nbytes + 8, None) == -1             # stride % 16
    assert run(f, f, f, None, None, None, 1, 256, 256, 256, g, s16 + 4, nbytes, None) == -1             # misaligned
    assert run(f, f, f, None, None, None, -1, 256, 256, 256, g, s16, nbytes, None) == -1
    assert run(f, f, f, None, None, None, 1, 256, 128, 256, g, s16, nbytes, None) == -1                 # in_stride < L
    assert run(None, f, f, None, None, None, 1, 256, 256, 256, g, s16, nbytes, None) == -1
    assert run(f, f, f, None, None, None, 0, 256, 256, 256, g, s16, nbytes, None) == 0                  # empty batch
    init = lib.aec_stage1_state_init
    assert init(None, 1, nbytes, None, g, None) == -1
    assert init(s16, 1, nbytes - 16, None, g, None) == -1
    assert init(s16, -1, nbytes, None, g, None) == -1
    assert init(s16, 0, nbytes, None, g, None) == 0
    assert A.launch_count() == 0


_ALGO = {"kAlgoPbfdaf": 2, "kAlgoPbfkf": 3}


def _expected_stream_builds():
    return sorted((2 if P <= 4 else P // 2, P, algo, echo, 128) for P in PS for algo in ALGOS for echo in (False, True))


def test_stream_unit_builds_the_twenty_kernels():
    with open(os.path.join(CSRC, "stage1_inst_ols_stream.cu")) as fh:
        text = re.sub(r"//[^\n]*", "", fh.read())
    rows = re.findall(r"AEC_STAGE1_BUILD\(\s*(\d+)\s*,\s*(\d+)\s*,\s*(\w+)\s*,\s*(true|false)\s*,\s*(\d+)\s*\)", text)
    got = sorted((int(nw), int(P), _ALGO[a], e == "true", int(r)) for nw, P, a, e, r in rows)
    assert got == _expected_stream_builds()


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
BUILDS = [(P, algo, echo) for P in PS for algo in ALGOS for echo in (False, True)]


def _bid(b):
    return f"P{b[0]}-{'kalman' if b[1] == 3 else 'nlms'}-{'echo' if b[2] else 'noecho'}"


def _torch():
    import torch
    return torch


def _cfg(P, algo, **kw):
    import acoustic_echo_cancellation_b200 as A
    return A.Stage1Config(partitions=P, algo=algo, **kw)


class _Raw:
    """Direct aec_stage1_run_stream calls on B streams (the C ABI, without Stage1Stream's pending samples)."""

    def __init__(self, B, cfg):
        import acoustic_echo_cancellation_b200 as A
        self.torch = _torch()
        self.cfg = cfg
        self.s = A.Stage1Stream(B, cfg)
        self.lib = _lib.load()

    def call(self, far, mic, ns, echo=False, erle=False, unaligned=False):
        """far, mic: numpy [B, L]; ns: samples per row (the kernel consumes ns // 256 blocks)"""
        torch = self.torch
        B, L = far.shape
        stride = L + 1 if unaligned else (L + 3) // 4 * 4
        off = 1 if unaligned else 0
        buf = torch.zeros((2, B * stride + 8), dtype=torch.float32, device="cuda")
        for i, x in enumerate((far, mic)):
            v = buf[i, off:off + B * stride].view(B, stride)
            v[:, :L] = torch.from_numpy(np.ascontiguousarray(x)).cuda()
        err = torch.full((B, stride + 4), 7.0, device="cuda")           # canary beyond L
        ech = torch.full((B, stride + 4), 7.0, device="cuda") if echo else None
        er = torch.zeros(B, device="cuda") if erle else None
        n_t = torch.as_tensor(np.asarray(ns, dtype=np.int64), device="cuda")
        c = self.cfg.to_c()
        rc = self.lib.aec_stage1_run_stream(buf[0, off:].data_ptr(), buf[1, off:].data_ptr(), err.data_ptr(),
                                            ech.data_ptr() if echo else None, er.data_ptr() if erle else None,
                                            n_t.data_ptr(), B, L, stride, stride + 4, C.byref(c),
                                            self.s.state.data_ptr(), self.s.state_stride,
                                            int(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc, "aec_stage1_run_stream")
        torch.cuda.synchronize()
        assert (err[:, L:] == 7.0).all(), "written past L"
        return err[:, :L].cpu().numpy(), None if ech is None else ech[:, :L].cpu().numpy(), \
            None if er is None else er.cpu().numpy()


def _schedules(P, B, nblk, rng):
    """per stream, a list of sample counts per call: 0-block and 1-block calls, every T0 residue mod P, odd and even
    block counts, and samples beyond the last whole block that the caller keeps"""
    out = []
    for b in range(B):
        sched, done = [], 0
        while done < nblk:
            if b == 0:
                k = 1 if len(sched) % 5 else 0
            elif b == 1:
                k = 3
            else:
                k = int(rng.choice([0, 1, 2, 5, 7, 16]))
            k = min(k, nblk - done)
            sched.append(k * H + int(rng.integers(0, H)))
            done += k
        out.append(sched)
    return out


def _chunked(raw, far, mic, scheds, echo=False, unaligned=False):
    B = far.shape[0]
    pos = [0] * B
    errs, echs = [[] for _ in range(B)], [[] for _ in range(B)]
    for k in range(max(len(s) for s in scheds)):
        ns = [s[k] if k < len(s) else 0 for s in scheds]
        L = max(max(ns), 1)
        fk = np.zeros((B, L), np.float32)
        mk = np.zeros((B, L), np.float32)
        for b in range(B):
            m = min(ns[b], far.shape[1] - pos[b])
            fk[b, :m] = far[b, pos[b]:pos[b] + m]
            mk[b, :m] = mic[b, pos[b]:pos[b] + m]
        e, y, _ = raw.call(fk, mk, ns, echo=echo, unaligned=unaligned)
        for b in range(B):
            used = ns[b] // H * H
            assert not e[b, used:].any()
            errs[b].append(e[b, :used])
            if echo:
                echs[b].append(y[b, :used])
            pos[b] += used
    return [np.concatenate(x) for x in errs], ([np.concatenate(x) for x in echs] if echo else None), pos


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
NBLK = 40


@pytest.mark.gpu
@pytest.mark.parametrize("b", BUILDS, ids=_bid)
def test_chunked_equals_one_call_bit_for_bit(b):
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    P, algo, echo = b
    B = 4
    far, mic = _signals(B, NBLK * H, 100 + P + algo)
    cfg = _cfg(P, algo)
    raw = _Raw(B, cfg)
    scheds = _schedules(P, B, NBLK, np.random.default_rng(P + 3 * algo))
    assert any(len(s) >= P for s in scheds)
    errs, echs, pos = _chunked(raw, far, mic, scheds, echo=echo)
    want = A.stage1_aec(torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda(), cfg, return_echo=echo)
    want_e = (want[0] if echo else want).cpu().numpy()
    for r in range(B):
        assert pos[r] == NBLK * H
        assert np.array_equal(errs[r], want_e[r, :NBLK * H]), f"stream {r}: err differs"
        if echo:
            assert np.array_equal(echs[r], want[1].cpu().numpy()[r, :NBLK * H]), f"stream {r}: echo differs"
    assert raw.s.state_views()["blocks"].cpu().tolist() == [NBLK] * B


@pytest.mark.gpu
def test_chunked_equals_one_call_with_unaligned_rows():
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    P, algo = 4, 3
    B = 3
    far, mic = _signals(B, NBLK * H, 7)
    cfg = _cfg(P, algo)
    raw = _Raw(B, cfg)
    scheds = _schedules(P, B, NBLK, np.random.default_rng(11))
    errs, _, _ = _chunked(raw, far, mic, scheds, unaligned=True)
    want = A.stage1_aec(torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda(), cfg).cpu().numpy()
    for r in range(B):
        assert np.array_equal(errs[r], want[r, :NBLK * H])


def _assert_fresh(s, rows, c0):
    """rows of Stage1Stream s as state_init leaves them: C = c0 exactly (Kalman step), every other field zero"""
    for name, t in s.state_views().items():
        v = t[rows].cpu().numpy()
        if name == "C":
            assert (v == np.float32(c0)).all(), f"C after init: {np.unique(v)[:4]} != {c0}"
        else:
            assert not v.any(), f"{name} is not zero after init"


@pytest.mark.gpu
@pytest.mark.parametrize("pset", (0, 1))
@pytest.mark.parametrize("P", (1, 4, 16))
@pytest.mark.parametrize("algo", ALGOS)
def test_chunked_at_non_default_parameters(algo, P, pset):
    """every other test of the stream kernel runs the default parameters, where a state init that ignored
    kalman_c0 (the stream kernel reads C from the state) would pass: chunked runs at the PARAMS sets equal one
    stage1_aec call bit for bit (error and echo), and the float64 oracle at 1e-4; the state right after state_init and
    after reset by indices and by bool mask is zero except C = kalman_c0"""
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    params = PARAMS[algo][pset]
    B = 4
    far, mic = _signals(B, NBLK * H, 800 + P + algo)
    cfg = _cfg(P, algo, **params)
    c0 = cfg.kalman_c0
    raw = _Raw(B, cfg)
    _assert_fresh(raw.s, list(range(B)), c0)
    scheds = _schedules(P, B, NBLK, np.random.default_rng(P + 3 * algo + 7 * pset))
    errs, echs, pos = _chunked(raw, far, mic, scheds, echo=True)
    want_e, want_y = (t.cpu().numpy() for t in A.stage1_aec(torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda(),
                                                            cfg, return_echo=True))
    cfg_o = O.AecConfig(partitions=P, algo=algo, **params)
    for r in range(B):
        assert pos[r] == NBLK * H
        assert np.array_equal(errs[r], want_e[r, :NBLK * H]), f"stream {r}: err differs"
        assert np.array_equal(echs[r], want_y[r, :NBLK * H]), f"stream {r}: echo differs"
        e64, y64 = O.pbfdaf_ols(far[r], mic[r], cfg_o)
        assert np.abs(errs[r] - e64).max() <= 1e-4
        assert np.abs(echs[r] - y64).max() <= 1e-4
    before = raw.s.state.clone()
    raw.s.reset([1, 3])
    _assert_fresh(raw.s, [1, 3], c0)
    raw.s.reset(torch.tensor([True, False, False, False]))
    _assert_fresh(raw.s, [0, 1, 3], c0)
    assert torch.equal(raw.s.state[2], before[2]), "reset touched a row it was not given"


def _call_kind(T0, k, skip):
    """where a call of k blocks from stream block T0 lies against the ERLE skip"""
    if k == 0:
        return "zero"
    if T0 + k <= skip:
        return "before"
    return "after" if T0 >= skip else "across"


# per stream, blocks per call: one block at a time (every boundary exactly), calls that straddle 5 and 13 or end / start
# on them, one call over everything
ERLE_BLOCKS = [[0] + [1] * 15 + [0, 5, 10], [3, 4, 0, 10, 13], [5, 8, 0, 17], [30]]
# Stage1Stream: one chunk length per call for all streams; blocks per call 0 3 0 1 4 0 7 5 12 1 0 16
ERLE_CHUNKS = [100, 700, 1, 255, 1000, 0, 2000, 1300, 3000, 333, 0, 4096]


def _check_erle(got, mic, e64, T0, k, skip, what):
    """got against O.erle_db over the call's blocks (stream blocks T0 .. T0 + k - 1) with index >= skip, within 0.05 dB;
    exactly 0 dB without any"""
    a = max(skip - T0, 0)
    if a >= k:
        assert got == 0.0, f"{what}, blocks {T0}+{k}, skip {skip}: {got} dB, want exactly 0"
    else:
        want = float(O.erle_db(mic[a * H:k * H], e64[a * H:k * H])[0])
        assert abs(got - want) <= 0.05, f"{what}, blocks {T0}+{k}, skip {skip}: {got} dB vs {want}"


@pytest.mark.gpu
@pytest.mark.parametrize("skip", (0, 5, 13))
def test_stream_erle_covers_the_blocks_from_the_skip(skip):
    """erle_db of every call covers the call's blocks whose index in the stream is >= erle_skip_hops (the only kernel
    that clamps erle_skip_hops - T0): calls wholly before the skip, across it, wholly after it and without a block,
    against the float64 oracle (chunked pbfdaf_ols_stream) within 0.05 dB, and exactly 0 dB where no block counts.
    Once through the C ABI with per-stream schedules, once through Stage1Stream.process(return_echo, return_erle),
    whose n_out, error, echo and ERLE must equal raw calls over the same blocks."""
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    P, algo = 8, 3
    cfg = _cfg(P, algo, erle_skip_hops=skip)
    cfg_o = O.AecConfig(partitions=P, algo=algo)
    B = len(ERLE_BLOCKS)
    nblk = sum(ERLE_CHUNKS) // H
    far, mic = _signals(B, (nblk + 1) * H, 900 + skip)
    rng = np.random.default_rng(skip)
    kinds = set()

    # the C ABI, a schedule per stream (samples past the last whole block are given and not consumed)
    raw = _Raw(B, cfg)
    T0, states = [0] * B, [None] * B
    for c in range(max(len(s) for s in ERLE_BLOCKS)):
        ks = [s[c] if c < len(s) else 0 for s in ERLE_BLOCKS]
        ns = [k * H + int(rng.integers(0, H)) for k in ks]
        L = max(ns)
        fk = np.zeros((B, L), np.float32)
        mk = np.zeros((B, L), np.float32)
        for b in range(B):
            fk[b, :ns[b]] = far[b, T0[b] * H:T0[b] * H + ns[b]]
            mk[b, :ns[b]] = mic[b, T0[b] * H:T0[b] * H + ns[b]]
        e, _, erle = raw.call(fk, mk, ns, erle=True)
        for b in range(B):
            k = ks[b]
            e64, _, states[b] = pbfdaf_ols_stream(fk[b, :k * H], mk[b, :k * H], cfg_o, states[b])
            assert np.abs(e[b, :k * H] - e64).max(initial=0.0) <= 1e-4
            _check_erle(erle[b], mk[b], e64, T0[b], k, skip, f"stream {b}")
            kinds.add(_call_kind(T0[b], k, skip))
            T0[b] += k
    assert kinds == ({"zero", "after"} if skip == 0 else {"zero", "before", "across", "after"})

    # Stage1Stream, the same chunks for every stream, against raw calls over the blocks each call consumes
    s = A.Stage1Stream(B, cfg)
    ref = _Raw(B, cfg)
    ft, mt = torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda()
    pos, T, kinds, states = 0, 0, set(), [None] * B
    for n in ERLE_CHUNKS:
        err, n_out, echo, erle = s.process(ft[:, pos:pos + n], mt[:, pos:pos + n], return_echo=True, return_erle=True)
        k = (pos + n) // H - T
        assert n_out.cpu().tolist() == [k * H] * B
        assert err.shape[1] >= k * H and echo.shape == err.shape
        e, y, erle_r = ref.call(far[:, T * H:(T + k) * H], mic[:, T * H:(T + k) * H], [k * H] * B, echo=True,
                                erle=True)
        assert np.array_equal(err[:, :k * H].cpu().numpy(), e) and not err[:, k * H:].any()
        assert np.array_equal(echo[:, :k * H].cpu().numpy(), y), "Stage1Stream's echo differs from the raw call's"
        assert np.array_equal(erle.cpu().numpy(), erle_r)
        for b in range(B):
            e64, _, states[b] = pbfdaf_ols_stream(far[b, T * H:(T + k) * H], mic[b, T * H:(T + k) * H], cfg_o, states[b])
            _check_erle(erle_r[b], mic[b, T * H:], e64, T, k, skip, f"Stage1Stream, stream {b}")
        kinds.add(_call_kind(T, k, skip))
        pos, T = pos + n, T + k
    assert kinds == ({"zero", "after"} if skip == 0 else {"zero", "before", "across", "after"})


def _occupancy_signals(B, n, seed):
    """B rows: 8 synthetic utterances, each row one of them at its own gain"""
    rng = np.random.default_rng(seed)
    far, mic = _signals(8, n, seed)
    g = (0.25 + 0.75 * rng.random(B)).astype(np.float32)[:, None]
    idx = np.arange(B) % 8
    return far[idx] * g, mic[idx] * g


@pytest.mark.gpu
@pytest.mark.parametrize("P,algo,Bspec", [(4, 3, (16, 5)), (16, 2, (4, 3))], ids=("P4-kalman-16sms+5", "P16-nlms-4sms+3"))
def test_full_occupancy_chunked_equals_one_call(P, algo, Bspec):
    """several full waves of co-resident CTAs (the two-warp build picks the warp that starts the transform chain from
    the hardware warp slot, which only varies when CTAs share an SM), each row its own ragged schedule: every row equals
    stage1_aec on the same rows bit for bit, two identical runs give identical outputs and stored state, and 16 random
    rows match the float64 oracle at 1e-4"""
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    B, nblk = Bspec[0] * sms + Bspec[1], 24
    far, mic = _occupancy_signals(B, nblk * H, 1000 + P)
    cfg = _cfg(P, algo)
    scheds = _schedules(P, B, nblk, np.random.default_rng(P))
    runs = []
    for _ in range(2):
        raw = _Raw(B, cfg)
        errs, _, pos = _chunked(raw, far, mic, scheds)
        assert pos == [nblk * H] * B
        runs.append((errs, raw.s.state.cpu().numpy()))
    assert all(np.array_equal(a, b) for a, b in zip(runs[0][0], runs[1][0])), "two identical runs differ"
    assert np.array_equal(runs[0][1], runs[1][1]), "two identical runs store different states"
    want = A.stage1_aec(torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda(), cfg).cpu().numpy()
    bad = [r for r in range(B) if not np.array_equal(runs[0][0][r], want[r])]
    assert not bad, f"{len(bad)} rows differ from stage1_aec, first {bad[:8]}"
    cfg_o = O.AecConfig(partitions=P, algo=algo)
    for r in np.random.default_rng(B).choice(B, size=16, replace=False):
        e64, _ = O.pbfdaf_ols(far[r], mic[r], cfg_o)
        assert np.abs(runs[0][0][r] - e64).max() <= 1e-4, f"row {r}"


def _oracle_state(far, mic, cfg_o, k, dtype=np.float64):
    _, _, st = pbfdaf_ols_stream(far[:k * H], mic[:k * H], cfg_o, None, dtype)
    return st


@pytest.mark.gpu
@pytest.mark.parametrize("P", PS)
@pytest.mark.parametrize("algo", ALGOS)
def test_state_matches_the_float64_oracle(P, algo):
    """every field after k blocks within 10x the float32 oracle's drift from the float64 one (relative to the field's
    largest magnitude in the row; the drift is measured here, on the same rows).  The drift counts as at least 1e-7:
    numpy runs the float32 oracle's transforms in float64 and rounds once (X drifts by 2-5e-8 on these rows, W by 3e-7
    with the NLMS step and 1.6-2.7e-6 with the Kalman step, Psi / C by 0.7-7e-6)."""
    B, k = 2, 37
    far, mic = _signals(B, k * H, 200 + P + algo)
    raw = _Raw(B, _cfg(P, algo))
    raw.call(far, mic, [k * H] * B)
    got = {n: v.cpu().numpy() for n, v in raw.s.state_views().items()}
    cfg_o = O.AecConfig(partitions=P, algo=algo)
    for r in range(B):
        s64 = _oracle_state(far[r], mic[r], cfg_o, k)
        s32 = _oracle_state(far[r], mic[r], cfg_o, k, np.float32)
        assert got["blocks"][r] == k
        assert np.array_equal(got["prev"][r], far[r, (k - 1) * H:k * H])
        for name in [n for n in got if n not in ("blocks", "prev")]:
            ref = np.asarray(s64[name])
            scale = max(np.abs(ref).max(), 1e-30)
            drift = np.abs(np.asarray(s32[name]) - ref).max() / scale
            err = np.abs(got[name][r] - ref).max() / scale
            assert err <= 10 * max(drift, 1e-7), f"{name} row {r}: {err:.3g} > 10 x {drift:.3g}"


@pytest.mark.gpu
@pytest.mark.parametrize("P", (1, 4, 16))
@pytest.mark.parametrize("algo", ALGOS)
def test_warm_start_from_the_oracle_state(P, algo):
    """the load path alone: the oracle's float64 state at block k, cast to float32, continued by the kernel"""
    torch = _torch()
    B, k, n = 2, 23, 30
    far, mic = _signals(B, n * H, 300 + P + algo)
    cfg_o = O.AecConfig(partitions=P, algo=algo)
    raw = _Raw(B, _cfg(P, algo, erle_skip_hops=0))
    v = raw.s.state_views()
    refs = []
    for r in range(B):
        st = _oracle_state(far[r], mic[r], cfg_o, k)
        for name, t in v.items():
            dt = {torch.int64: np.int64, torch.complex64: np.complex64, torch.float32: np.float32}[t.dtype]
            t[r] = torch.as_tensor(np.asarray(st[name]).astype(dt), device="cuda")
        e, _, _ = pbfdaf_ols_stream(far[r, k * H:], mic[r, k * H:], cfg_o, st)
        refs.append(e)
    err, _, erle = raw.call(far[:, k * H:], mic[:, k * H:], [(n - k) * H] * B, erle=True)
    for r in range(B):
        assert np.abs(err[r] - refs[r]).max() <= 1e-4
        want = O.erle_db(mic[r, k * H:], refs[r])[0]
        assert abs(erle[r] - want) <= 0.05


@pytest.mark.gpu
@pytest.mark.parametrize("chunk", (160, 1, 333))
def test_stage1_stream_any_chunk_length(chunk):
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    B, n = 3, (12 if chunk == 1 else 40) * H + 77
    far, mic = _signals(B, n, 400 + chunk)
    cfg = _cfg(4, 2)
    s = A.Stage1Stream(B, cfg)
    outs = [[] for _ in range(B)]
    ft, mt = torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda()
    for pos in range(0, n, chunk):
        e, n_out = s.process(ft[:, pos:pos + chunk], mt[:, pos:pos + chunk])
        n_out = n_out.cpu().tolist()
        assert not e[:, max(n_out):].any()
        for r in range(B):
            outs[r].append(e[r, :n_out[r]])
    want = A.stage1_aec(ft, mt, cfg)
    m = n // H * H
    for r in range(B):
        assert torch.equal(torch.cat(outs[r]), want[r, :m])


@pytest.mark.gpu
def test_stage1_stream_reset_rows():
    import acoustic_echo_cancellation_b200 as A
    torch = _torch()
    B, n, cut = 4, 30 * H, 11 * H + 100
    far, mic = _signals(B, n, 500)
    ft, mt = torch.from_numpy(far).cuda(), torch.from_numpy(mic).cuda()
    cfg = _cfg(8, 3)
    s = A.Stage1Stream(B, cfg)
    before = [s.process(ft[:, :cut], mt[:, :cut])]
    s.reset([1, 3])
    after = [s.process(ft[:, cut:], mt[:, cut:])]
    whole = A.stage1_aec(ft, mt, cfg)
    fresh = A.stage1_aec(ft[:, cut:].contiguous(), mt[:, cut:].contiguous(), cfg)
    for r in range(B):
        got = torch.cat([after[0][0][r, :after[0][1][r]]])
        if r in (1, 3):
            m = (n - cut) // H * H
            assert torch.equal(got, fresh[r, :m])
        else:
            prev = before[0][0][r, :before[0][1][r]]
            assert torch.equal(torch.cat([prev, got]), whole[r, :n // H * H])


@pytest.mark.gpu
def test_batch_and_call_hygiene():
    torch = _torch()
    P, algo = 4, 2
    cfg = _cfg(P, algo)
    far, mic = _signals(3, 9 * H, 600)
    # a row alone equals the same row in a batch; repeated runs give the same bits
    runs = []
    for _ in range(2):
        raw = _Raw(3, cfg)
        runs.append([raw.call(far, mic, [9 * H, 5 * H + 3, 7 * H], erle=True),
                     raw.call(far, mic, [2 * H, 4 * H, 0], erle=True)])
    for a, b in zip(*runs):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])
    alone = _Raw(1, cfg)
    e1, _, _ = alone.call(far[1:2], mic[1:2], [5 * H + 3])
    assert np.array_equal(e1[0], runs[0][0][0][1])
    # a call without a whole block leaves the state bytes untouched; canaries past state_bytes stay
    raw = _Raw(2, cfg)
    raw.call(far[:2], mic[:2], [3 * H, 2 * H])
    big = _Raw(2, cfg)
    stride = big.s.state_stride + 64
    st = torch.full((2, stride), 0xA5, dtype=torch.uint8, device="cuda")
    st[:, :big.s.state_bytes] = raw.s.state
    big.s.state, big.s.state_stride = st, stride
    before = st.clone()
    big.call(far[:2], mic[:2], [255, 0])
    assert torch.equal(st, before)
    big.call(far[:2], mic[:2], [H, 0])
    assert torch.equal(st[1], before[1]) and not torch.equal(st[0], before[0])
    assert (st[:, big.s.state_bytes:] == 0xA5).all()
    # state_init: masked-out rows and the bytes past state_bytes stay untouched
    lib = _lib.load()
    c = cfg.to_c()
    st.fill_(0xA5)
    mask = torch.tensor([0, 1], dtype=torch.uint8, device="cuda")
    assert lib.aec_stage1_state_init(st.data_ptr(), 2, stride, mask.data_ptr(), C.byref(c),
                                     int(torch.cuda.current_stream().cuda_stream)) == 0
    torch.cuda.synchronize()
    assert (st[0] == 0xA5).all()
    assert not st[1, :big.s.state_bytes].any() and (st[1, big.s.state_bytes:] == 0xA5).all()


def _template_args(name):
    m = re.search(r"stage1_ols_stream_kernel<([^<>]*)>", name)
    if not m:
        return None
    norm = {"1u": "1", "0u": "0", "true": "1", "false": "0"}
    return [norm.get(a, a) for a in (re.sub(r"^\(\w+\)", "", a.strip()) for a in m.group(1).split(","))]


@pytest.mark.gpu
def test_profiler_names_the_stream_kernel():
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    far, mic = _signals(1, 4 * H, 700)
    wrong = []
    for P, algo, echo in BUILDS:
        raw = _Raw(1, _cfg(P, algo))
        raw.call(far, mic, [4 * H], echo=echo)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            raw.call(far, mic, [4 * H], echo=echo)
        names = {e.name for e in prof.events() if "stage1_ols_stream_kernel" in e.name}
        want = [str(P), "1" if algo == 3 else "0", "1" if echo else "0", "128"]
        if len(names) != 1 or _template_args(next(iter(names))) != want:
            wrong.append((P, algo, echo, sorted(names)))
    assert not wrong, wrong
