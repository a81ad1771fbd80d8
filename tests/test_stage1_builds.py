"""Every compiled stage-1 kernel build against the float64 oracle (oracle/aec_oracle.py).

``BUILDS`` lists each instantiation of the eight ``stage1_inst_*.cu`` units with the ``aec_cfg.variant`` that selects
it; a CPU test keeps the table equal to what those units instantiate.  The GPU tests (-m gpu) then run

  * every build on a ragged batch whose lengths sit on its chunk edges (error signal, echo estimate, ERLE, the zeros
    beyond each utterance; features for the fused-feature builds) and check, with the profiler, that the launch ran the
    kernel the table names;
  * the no-echo / echo twins of a build and ``variant = 0`` against the build the library documents as the default,
    bit for bit;
  * the combinations the dispatch must refuse (nothing launched, nothing written);
  * one build per code path at non-default filter parameters, on far ends that are single tones at the special bins
    (DC, Nyquist, the self-mirrored bin N / 4 and their neighbours), and at signal levels down to 1 LSB of 16-bit PCM
    with a bar relative to the level.

Bars: 1e-4 max-abs on the error signal and the echo estimate, 0.05 dB on ERLE, features 2e-5 x max(1, max|ref|) against
``stage2_features`` of the kernel's own error signal.  The level test adds 1e-4 x max|mic| per row.
"""
import ctypes as C
import functools
import os
import re
from collections import namedtuple

import numpy as np
import pytest

from oracle import aec_oracle as O

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "acoustic_echo_cancellation_b200", "csrc")

TOL_ERR = 1e-4       # max abs, error signal and echo estimate
TOL_ERLE = 0.05      # dB
TOL_FEAT = 2e-5      # x max(1, max|ref|), fused features against stage2_features of the stored error signal
SKIP = 8             # erle_skip_hops

NLMS, KALMAN, OLS_NLMS, OLS_KALMAN = 0, 1, 2, 3

# entry: the stage1_inst_<entry>.cu unit; warps per utterance; regs: register cap (__maxnreg__); variant: the
# aec_cfg.variant that selects the build (0 where the entry takes none: the frame-1024 overlap-save kernels and the
# fused-feature builds, which are chosen from P, algo and the batch size)
Build = namedtuple("Build", "entry frame P algo echo warps regs variant")


def _stft(entry, warps, rows, frame=512):
    return [Build(entry, frame, P, algo, echo, warps, regs, 1000 * warps + regs) for (P, algo, echo, regs) in rows]


def _ols(P, regs_nlms, regs_kal):
    warps = 2 if P <= 4 else P // 2
    return [Build("ols", 512, P, algo, echo, warps, regs, 1000 * warps + regs)
            for algo, regs in ((OLS_NLMS, regs_nlms), (OLS_KALMAN, regs_kal)) for echo in (False, True)]


BUILDS = (
    _stft("nw1", 1, [(4, NLMS, False, 255), (4, NLMS, False, 200)])
    + _stft("nw2", 2, [(4, NLMS, False, 128), (4, NLMS, False, 168), (4, NLMS, True, 168),
                       (4, KALMAN, False, 168), (4, KALMAN, False, 128), (4, KALMAN, True, 200),
                       (1, NLMS, False, 128), (1, NLMS, True, 128), (1, KALMAN, False, 128), (1, KALMAN, True, 128),
                       (2, NLMS, False, 128), (2, NLMS, True, 128), (2, KALMAN, False, 128), (2, KALMAN, True, 128)])
    + _stft("nw4", 4, [(8, NLMS, False, 128), (8, NLMS, False, 168), (8, NLMS, True, 168),
                       (8, KALMAN, False, 168), (8, KALMAN, True, 168),
                       (16, NLMS, False, 255), (16, NLMS, True, 255), (16, KALMAN, False, 255), (16, KALMAN, True, 255),
                       (4, NLMS, False, 128), (4, NLMS, False, 96)])
    + _stft("nw8", 8, [(P, algo, echo, 128) for P in (16, 8) for algo in (KALMAN, NLMS) for echo in (False, True)])
    + _stft("1024", 8, [(P, algo, echo, 128) for P in (8, 4, 2, 1) for algo in (NLMS, KALMAN) for echo in (False, True)],
            frame=1024)
    + _ols(4, 128, 128) + _ols(4, 128, 168)[2:] + _ols(4, 168, 168)[:2]
    + _ols(1, 128, 128) + _ols(2, 128, 128) + _ols(8, 128, 128) + _ols(16, 128, 128)
    + [Build("ols1024", 1024, P, algo, echo, P, 128, 0) for P in (8, 4) for algo in (OLS_NLMS, OLS_KALMAN)
       for echo in (False, True)]
    + [Build("feat", 512, 4, NLMS, False, 2, 168, 0), Build("feat", 512, 4, NLMS, False, 2, 200, 0),
       Build("feat", 512, 4, KALMAN, False, 2, 200, 0), Build("feat", 512, 2, NLMS, False, 2, 168, 0),
       Build("feat", 512, 1, NLMS, False, 2, 168, 0)]
)

ALGO_NAMES = {NLMS: "nlms", KALMAN: "kalman", OLS_NLMS: "ols-nlms", OLS_KALMAN: "ols-kalman"}


def _bid(b):
    return f"{b.entry}-P{b.P}-{ALGO_NAMES[b.algo]}-{'echo' if b.echo else 'noecho'}-r{b.regs}"


# variant = 0: the build each (frame, P, algo, echo) runs by default (the first instantiation listed for it in
# stage1_inst_nw2.cu / nw8.cu: two warps at P <= 4 -- 128 registers, 168 for NLMS with the echo output and for Kalman
# without it, 200 for Kalman with it --, eight warps from P = 8; the overlap-save kernels at 128 registers)
def _default_variant(frame, P, algo, echo):
    if algo in (OLS_NLMS, OLS_KALMAN):
        return 1000 * (2 if P <= 4 else P // 2) + 128
    if frame == 1024 or P >= 8:
        return 8128
    if P == 4:
        return {(NLMS, False): 2128, (NLMS, True): 2168, (KALMAN, False): 2168, (KALMAN, True): 2200}[(algo, echo)]
    return 2128


DEFAULTS = sorted({(b.frame, b.P, b.algo, b.echo) for b in BUILDS if b.entry not in ("feat", "ols1024")})


# ---------------------------------------------------------------------------------------------------------------------
# a. the table and what the units instantiate (CPU)
# ---------------------------------------------------------------------------------------------------------------------
_ALGO_TOKENS = {"kAlgoNlms": NLMS, "kAlgoKalman": KALMAN, "kAlgoPbfdaf": OLS_NLMS, "kAlgoPbfkf": OLS_KALMAN}


def _instantiations():
    """Every (entry, frame, P, algo, echo, warps, regs) the stage1_inst_*.cu units compile, read from their
    AEC_STAGE1_BUILD(NW, P, ALGO, ECHO, REGS) lines."""
    found = set()
    for unit in ("nw1", "nw2", "nw4", "nw8", "1024", "feat", "ols", "ols1024"):
        with open(os.path.join(CSRC, f"stage1_inst_{unit}.cu")) as f:
            text = re.sub(r"//[^\n]*", "", f.read())      # (builds named in comments do not count)
        builds = re.findall(r"AEC_STAGE1_BUILD\(\s*(\d+)\s*,\s*(\d+)\s*,\s*(\w+)\s*,\s*(true|false)\s*,\s*(\d+)\s*\)", text)
        assert builds, f"no AEC_STAGE1_BUILD line in stage1_inst_{unit}.cu"
        for nw, P, algo, echo, regs in builds:
            frame = 1024 if unit in ("1024", "ols1024") else 512
            found.add((unit, frame, int(P), _ALGO_TOKENS[algo], echo == "true", int(nw), int(regs)))
    return found


def test_build_table_lists_every_instantiation():
    """BUILDS is exactly what the units compile: a build added without a table entry (so without a test) fails here,
    and so does a table entry whose build was removed."""
    table = [tuple(b)[:7] for b in BUILDS]
    assert len(table) == len(set(table)), "duplicate BUILDS entry"
    found = _instantiations()
    assert found - set(table) == set(), f"built but not in BUILDS: {sorted(found - set(table))}"
    assert set(table) - found == set(), f"in BUILDS but not built: {sorted(set(table) - found)}"
    assert len(BUILDS) == 88
    # the variant of a build names its warps and registers, except where the entry takes none
    for b in BUILDS:
        assert b.variant == (0 if b.entry in ("feat", "ols1024") else 1000 * b.warps + b.regs), b
    # every default names a build of the table
    for key in DEFAULTS:
        v = _default_variant(*key)
        assert any((b.frame, b.P, b.algo, b.echo, b.variant) == key + (v,) for b in BUILDS), (key, v)


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _A():
    import acoustic_echo_cancellation_b200 as A
    return A


def _cuda(x):
    return _torch().from_numpy(np.ascontiguousarray(x)).cuda()


@functools.lru_cache(maxsize=1)
def _erb():
    return _cuda(O.erb_filterbank().astype(np.float32))


def _sms():
    torch = _torch()
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def _hop(b):
    return b.frame // 2


def _chunk_frames(b):
    """hops a kernel stages per chunk: Stage1Smem<NW, P>::F (2 NW, 8 on the 16-partition ring kernel), 8 on the
    frame-1024 kernel; the overlap-save kernels work block by block from a ring of 4 staged far-end blocks"""
    if b.entry in ("ols", "ols1024"):
        return 4
    if b.entry == "1024":
        return 8
    if b.warps == 8 and b.P >= 16:
        return 8
    return 2 * b.warps


def _oracle_cfg(b, **params):
    return O.AecConfig(frame=b.frame, partitions=b.P, algo=b.algo, delta=params.pop("delta", 1e-6 * b.frame), **params)


def _zero_tails(far, mic, ns):
    """rows zero-padded beyond their length, as the reference's collate_fn pads a ragged batch"""
    far, mic = far.copy(), mic.copy()
    for i, n in enumerate(ns):
        far[i, n:] = 0
        mic[i, n:] = 0
    return far, mic


def _run(b, far, mic, ns=None, skip=SKIP, **params):
    """one launch of build b; returns numpy err, echo (or None), erle, feat (or None) and the device tensors of err and
    far (for the feature reference)"""
    A, torch = _A(), _torch()
    cfg = A.Stage1Config(frame=b.frame, partitions=b.P, algo=b.algo, erle_skip_hops=skip, variant=b.variant, **params)
    far_t = far if isinstance(far, torch.Tensor) else _cuda(far)
    mic_t = mic if isinstance(mic, torch.Tensor) else _cuda(mic)
    ns_t = None if ns is None else _cuda(np.asarray(ns, dtype=np.int64))
    echo = feat = None
    if b.entry == "feat":
        err, feat, erle = A.stage1_aec_features(far_t, mic_t, _erb(), cfg, n_samples=ns_t, return_erle=True)
    elif b.echo:
        err, echo, erle = A.stage1_aec(far_t, mic_t, cfg, n_samples=ns_t, return_echo=True, return_erle=True)
    else:
        err, erle = A.stage1_aec(far_t, mic_t, cfg, n_samples=ns_t, return_erle=True)
    torch.cuda.synchronize()
    return {"err": err.cpu().numpy(), "echo": None if echo is None else echo.cpu().numpy(), "erle": erle.cpu().numpy(),
            "feat": feat, "err_t": err, "far_t": far_t}


def _check(b, out, ref, lens, tol=TOL_ERR, rows=None):
    """out (of _run) against the oracle's ref for the given rows: error signal and echo estimate within tol (a scalar or
    one bar per row), exact zeros beyond each utterance's (n // hop) * hop output samples, ERLE within TOL_ERLE (the
    oracle gives 0 dB to an utterance no longer than the skipped hops, and so must the kernel); fused features against
    stage2_features of the kernel's own error signal"""
    rows = list(range(len(lens))) if rows is None else list(rows)
    tol = np.broadcast_to(np.asarray(tol, dtype=np.float64).reshape(-1, 1), (len(rows), 1))
    hop = _hop(b)
    n = ref["err"].shape[1]
    for name in ("err", "echo"):
        got = out[name]
        if got is None:
            continue
        got = got[rows]
        diff = np.abs(got[:, :n].astype(np.float64) - ref[name])
        worst = diff.max(axis=1, initial=0.0)
        assert (worst[:, None] <= tol).all(), f"{name}: max |kernel - oracle| per row {worst} > {tol.ravel()}"
        for i, r in enumerate(rows):
            m = (int(lens[r]) // hop) * hop
            assert not got[i, m:].any(), f"{name}: row {r} (n = {lens[r]}) is not zero beyond sample {m}"
    derle = np.abs(out["erle"][rows].astype(np.float64) - ref["erle_db"])
    assert derle.max() <= TOL_ERLE, f"ERLE: |kernel - oracle| per row {derle}"
    if out["feat"] is not None:
        A, torch = _A(), _torch()
        want = A.stage2_features(out["err_t"], out["far_t"], _erb(), in_norm=False)
        silent = A.stage2_features(torch.zeros(1, 512, device="cuda"), torch.zeros(1, 512, device="cuda"), _erb(),
                                   in_norm=False)[0, 0]
        feat = out["feat"]
        for r in rows:
            tb = O.n_frames(int(lens[r]), b.frame, hop)
            w = want[r, :tb]
            bar = TOL_FEAT * max(1.0, float(w.abs().max()) if tb else 0.0)
            d = float((feat[r, :tb] - w).abs().max()) if tb else 0.0
            assert d <= bar, f"features of row {r}: {d} > {bar}"
            if tb < feat.shape[1]:
                d = float((feat[r, tb:] - silent).abs().max())
                assert d <= TOL_FEAT * max(1.0, float(silent.abs().max())), f"features beyond row {r}'s frames: {d}"


# ---------------------------------------------------------------------------------------------------------------------
# b. every build on its chunk edges
# ---------------------------------------------------------------------------------------------------------------------
L_LONG = 16000 + 123


@functools.lru_cache(maxsize=None)
def _signals(frame, P, first_u, B, L):
    d = synth_batch(first_u, B, L, frame, P)
    return d["far"], d["mic"], frame // 2


def synth_batch(first_u, B, L, frame, P):
    from acoustic_echo_cancellation_b200 import synth
    return synth.make_batch(first_u, B, L, sample_rate=16000 * frame // 512, rir_len=min(P * frame // 2, 4096))


@functools.lru_cache(maxsize=None)
def _ragged_case(frame, P, algo, chunk):
    """ragged inputs (tails zeroed) and their float64 oracle, shared by the builds of one (frame, P, algo, chunk)"""
    hop = frame // 2
    c = chunk * hop
    lens = np.array([0, 1, 255, 256, 257, c - 1, c, c + 1, L_LONG], dtype=np.int64)
    far, mic, _ = _signals(frame, P, 10 * P + algo, len(lens), L_LONG)
    far, mic = _zero_tails(far, mic, lens)
    b = Build("", frame, P, algo, False, 0, 0, 0)
    ref = O.stage1(far, mic, _oracle_cfg(b), n_samples=lens, erle_skip=SKIP * hop)
    return far, mic, lens, ref


@pytest.mark.gpu
@pytest.mark.parametrize("b", BUILDS, ids=_bid)
def test_build_matches_oracle_on_chunk_edges(b):
    """lengths 0, 1, 255, 256, 257, chunk - 1, chunk, chunk + 1 samples and 16 123 in one ragged batch (chunk: the hops a
    kernel stages at a time); the fused-feature build for many-wave batches is only selected from B = 20 x SM count, so
    its batch is the ragged rows plus copies of 16 more utterances at random gains, of which 16 are checked too, and its
    error signal must equal the plain kernel's bit for bit (as must every fused build's)"""
    torch = _torch()
    far, mic, lens, ref = _ragged_case(b.frame, b.P, b.algo, _chunk_frames(b))
    if b.entry == "feat" and b.regs == 168 and b.P == 4:
        Bn = 20 * _sms()
        base_f, base_m, _ = _signals(512, 4, 300, 16, L_LONG)
        rng = np.random.default_rng(5)
        gains = (0.25 + 0.75 * rng.random(Bn - len(lens))).astype(np.float32)
        idx = np.arange(Bn - len(lens)) % 16
        fill_f = _cuda(base_f)[_cuda(idx)] * _cuda(gains)[:, None]
        fill_m = _cuda(base_m)[_cuda(idx)] * _cuda(gains)[:, None]
        far_t = torch.cat([_cuda(far), fill_f])
        mic_t = torch.cat([_cuda(mic), fill_m])
        all_lens = np.concatenate([lens, np.full(Bn - len(lens), L_LONG, dtype=np.int64)])
        assert Bn >= 20 * _sms()
        out = _run(b, far_t, mic_t, all_lens)
        _check(b, out, ref, all_lens, rows=range(len(lens)))
        pick = np.sort(rng.choice(np.arange(len(lens), Bn), size=16, replace=False))
        ref16 = O.stage1(far_t[pick].cpu().numpy(), mic_t[pick].cpu().numpy(), _oracle_cfg(b), erle_skip=SKIP * 256)
        _check(b, out, ref16, all_lens, rows=pick)
    else:
        far_t, mic_t, all_lens = _cuda(far), _cuda(mic), lens
        out = _run(b, far_t, mic_t, lens)
        _check(b, out, ref, lens)
    if b.entry == "feat":
        A = _A()
        plain, erle = A.stage1_aec(far_t, mic_t, A.Stage1Config(partitions=b.P, algo=b.algo, erle_skip_hops=SKIP),
                                   n_samples=_cuda(all_lens), return_erle=True)
        assert torch.equal(out["err_t"], plain)
        assert np.array_equal(out["erle"], erle.cpu().numpy())


def _kernel_name(b):
    """(name, template arguments) of the __global__ function build b launches"""
    e = str(b.echo).lower()
    if b.entry in ("nw1", "nw2", "nw4", "nw8"):
        return "stage1_n512_kernel", [b.warps, b.P, b.algo, e, b.regs, "false"]
    if b.entry == "feat":
        return "stage1_n512_kernel", [b.warps, b.P, b.algo, e, b.regs, "true"]
    if b.entry == "1024":
        return "stage1_n1024_kernel", [b.P, b.algo, e, b.regs]
    kal = str(b.algo == OLS_KALMAN).lower()
    return ("stage1_ols_kernel" if b.entry == "ols" else "stage1_ols1024_kernel"), [b.P, kal, e, b.regs]


def _template_args(name, kernel):
    m = re.search(re.escape(kernel) + r"<([^<>]*)>", name)
    if not m:
        return None
    args = []
    for a in m.group(1).split(","):
        a = re.sub(r"^\(\w+\)", "", a.strip())        # "(bool)1" / "(int)4" forms of some demanglers
        a = {"1u": "1", "0u": "0"}.get(a, a)
        args.append(a)
    return args


def _norm(v):
    v = str(v)
    return {"true": "1", "false": "0"}.get(v, v)


@pytest.mark.gpu
def test_every_build_launches_the_kernel_it_names():
    """The profiler's record of each launch names the template instance the table gives: a dispatch that quietly ran
    another build (a different register cap, warp count or echo flag computes the same numbers) fails here."""
    torch = _torch()
    from torch.profiler import ProfilerActivity, profile
    d = {f: synth_batch(0, 1, 4096, f, 4) for f in (512, 1024)}

    def inputs(b):
        far, mic = _cuda(d[b.frame]["far"]), _cuda(d[b.frame]["mic"])
        if b.entry == "feat" and b.regs == 168 and b.P == 4:       # selected from B = 20 x SM count
            n = 20 * _sms()
            return far.expand(n, -1).contiguous(), mic.expand(n, -1).contiguous()
        return far, mic

    for b in BUILDS:                                     # first launches (attribute set-up) outside the profiler
        _run(b, *inputs(b))
    wrong = []
    for b in BUILDS:
        far, mic = inputs(b)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _run(b, far, mic)
            torch.cuda.synchronize()
        kernel, want = _kernel_name(b)
        names = {e.name for e in prof.events() if "stage1_" in e.name and "kernel" in e.name}
        got = [_template_args(n, kernel) for n in names]
        if len(names) != 1 or got[0] is None or [_norm(a) for a in got[0]] != [_norm(a) for a in want]:
            wrong.append((_bid(b), sorted(names)))
    assert not wrong, wrong


# ---------------------------------------------------------------------------------------------------------------------
# c. same build, same bits
# ---------------------------------------------------------------------------------------------------------------------
def _echo_twins():
    by_key = {}
    for b in BUILDS:
        if b.entry != "feat":
            by_key.setdefault((b.entry, b.frame, b.P, b.algo, b.warps, b.regs), {})[b.echo] = b
    return [(v[False], v[True]) for v in by_key.values() if len(v) == 2]


@functools.lru_cache(maxsize=None)
def _bitwise_case(frame, P):
    lens = np.array([L_LONG, L_LONG - 777, 4097, 300], dtype=np.int64)
    far, mic, _ = _signals(frame, P, 50 + P, len(lens), L_LONG)
    far, mic = _zero_tails(far, mic, lens)
    return far, mic, lens


@pytest.mark.gpu
@pytest.mark.parametrize("pair", _echo_twins(), ids=lambda p: _bid(p[0]).replace("-noecho", ""))
def test_echo_output_leaves_the_error_signal_bit_for_bit(pair):
    """a build with the echo-estimate output and its twin without it (same warps, P, algo, registers) compute the same
    error signal and ERLE, bit for bit"""
    far, mic, lens = _bitwise_case(pair[0].frame, pair[0].P)
    a, b = (_run(x, far, mic, lens) for x in pair)
    assert np.array_equal(a["err"], b["err"])
    assert np.array_equal(a["erle"], b["erle"])


@pytest.mark.gpu
@pytest.mark.parametrize("key", DEFAULTS, ids=lambda k: f"f{k[0]}-P{k[1]}-{ALGO_NAMES[k[2]]}-{'echo' if k[3] else 'noecho'}")
def test_variant_zero_is_the_documented_default(key):
    frame, P, algo, echo = key
    v = _default_variant(*key)
    far, mic, lens = _bitwise_case(frame, P)
    named = next(b for b in BUILDS if (b.frame, b.P, b.algo, b.echo, b.variant) == (frame, P, algo, echo, v))
    a = _run(named, far, mic, lens)
    d = _run(named._replace(variant=0), far, mic, lens)
    for k in ("err", "echo", "erle"):
        assert (a[k] is None and d[k] is None) or np.array_equal(a[k], d[k]), k


# ---------------------------------------------------------------------------------------------------------------------
# d. combinations that must be refused
# ---------------------------------------------------------------------------------------------------------------------
REFUSED = [
    # (what, entry, frame, P, algo, echo, variant)
    ("1-warp build has no echo output", "run", 512, 4, NLMS, True, 1255),
    ("1-warp builds are NLMS only", "run", 512, 4, KALMAN, False, 1255),
    ("no 200-register 4-warp build", "run", 512, 4, NLMS, False, 4200),
    ("no 3-warp kernel", "run", 512, 4, NLMS, False, 3128),
    ("bare register cap", "run", 512, 4, NLMS, False, 168),
    ("8 warps not built at P = 4", "run", 512, 4, NLMS, False, 8128),
    ("2 warps not built at P = 16", "run", 512, 16, KALMAN, False, 2128),
    ("frame 1024: no 168-register build", "run", 1024, 8, NLMS, False, 2168),
    ("frame 1024: 8 warps only", "run", 1024, 8, NLMS, False, 2128),
    ("frame 1024: 8 warps only (1-warp cap)", "run", 1024, 4, NLMS, False, 1255),
    ("overlap-save P = 4 runs 2 warps", "run", 512, 4, OLS_NLMS, False, 8128),
    ("overlap-save P = 4 runs 2 warps (Kalman)", "run", 512, 4, OLS_KALMAN, True, 4128),
    ("overlap-save P = 16 runs 8 warps", "run", 512, 16, OLS_KALMAN, False, 2128),
    ("overlap-save P = 8 runs 4 warps", "run", 512, 8, OLS_NLMS, True, 8128),
    ("overlap-save: bare register cap", "run", 512, 4, OLS_NLMS, False, 168),
    ("overlap-save P = 8: no 168-register build", "run", 512, 8, OLS_KALMAN, False, 4168),
    ("overlap-save frame 1024 takes no variant", "run", 1024, 8, OLS_NLMS, False, 8128),
    ("overlap-save frame 1024 takes no variant (P = 4)", "run", 1024, 4, OLS_KALMAN, True, 4128),
    ("fused features take no variant", "feat", 512, 4, NLMS, False, 2168),
    ("fused features take no variant (200)", "feat", 512, 4, NLMS, False, 2200),
    ("fused features take no variant (Kalman)", "feat", 512, 4, KALMAN, False, 2200),
    ("no fused features for overlap-save", "feat", 512, 4, OLS_NLMS, False, 0),
    ("no fused Kalman build at P = 2", "feat", 512, 2, KALMAN, False, 0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", REFUSED, ids=lambda c: c[0].replace(" ", "_"))
def test_unbuilt_combination_is_refused_without_a_launch(case):
    """AEC_EUNSUPPORTED (-2), no launch counted, every output buffer still holds its canary"""
    A, torch = _A(), _torch()
    from acoustic_echo_cancellation_b200 import _lib
    _, entry, frame, P, algo, echo, variant = case
    B, L, pad, canary = 3, 4096, 64, 12345.0
    d = synth_batch(0, B, L, frame, P)
    far, mic = _cuda(d["far"]), _cuda(d["mic"])
    stride = L + 2 * pad
    err = torch.full((B, stride), canary, device="cuda")
    ech = torch.full((B, stride), canary, device="cuda")
    erle = torch.full((B,), canary, device="cuda")
    feat = torch.full((B, O.n_frames(L, frame, frame // 2), 64), canary, device="cuda")
    c = A.Stage1Config(frame=frame, partitions=P, algo=algo, variant=variant).to_c()
    lib = _lib.load()
    stream = int(torch.cuda.current_stream().cuda_stream)
    lib.aec_init()
    before = lib.aec_launch_count(0)
    if entry == "feat":
        rc = lib.aec_stage1_run_features(far.data_ptr(), mic.data_ptr(), err[:, pad:].data_ptr(), erle.data_ptr(),
                                         feat.data_ptr(), _erb().data_ptr(), None, B, L, L, stride, C.byref(c), stream)
    else:
        rc = lib.aec_stage1_run(far.data_ptr(), mic.data_ptr(), err[:, pad:].data_ptr(),
                                ech[:, pad:].data_ptr() if echo else None, erle.data_ptr(), None, B, L, L, stride,
                                C.byref(c), stream)
    torch.cuda.synchronize()
    assert rc == -2
    assert lib.aec_launch_count(0) == before
    for t in (err, ech, erle, feat):
        assert bool((t == canary).all())


# ---------------------------------------------------------------------------------------------------------------------
# e-g. one build per code path: filter parameters, tones at the special bins, signal levels
# ---------------------------------------------------------------------------------------------------------------------
def _pick(entry, P, algo, regs=None, echo=None, frame=None):
    cands = [b for b in BUILDS if b.entry == entry and b.P == P and b.algo == algo and (regs is None or b.regs == regs)
             and (frame is None or b.frame == frame)]
    if echo is None:                                     # the echo twin where there is one: its output is checked too
        cands.sort(key=lambda b: not b.echo)
    else:
        cands = [b for b in cands if b.echo == echo]
    return cands[0]


# Every code path of the recurrence: the 1-warp (4 pairs per thread), 2-warp (2 pairs; P = 1 to 4), 4-warp (1 pair;
# registers at P = 16) kernels, the 8-warp one-bin-per-thread kernel at P = 8 and its shared-memory ring form at P = 16
# (bin N / 4 one chunk ahead), the frame-1024 kernel, the overlap-save kernels at P = 1, 4 (bin 128 serial) and 8, 16
# (bin 128 on P lanes), frame-1024 overlap-save, the fused-feature builds.
PATHS = [
    _pick("nw1", 4, NLMS, 255),
    _pick("nw2", 1, NLMS), _pick("nw2", 4, NLMS, 168), _pick("nw2", 4, KALMAN, 200),
    _pick("nw4", 4, NLMS, 128), _pick("nw4", 8, NLMS, 168), _pick("nw4", 8, KALMAN, 168),
    _pick("nw4", 16, NLMS, 255), _pick("nw4", 16, KALMAN, 255),
    _pick("nw8", 8, NLMS), _pick("nw8", 8, KALMAN), _pick("nw8", 16, NLMS), _pick("nw8", 16, KALMAN),
    _pick("1024", 8, NLMS), _pick("1024", 8, KALMAN), _pick("1024", 1, KALMAN),
    _pick("ols", 1, OLS_NLMS), _pick("ols", 4, OLS_NLMS, 128), _pick("ols", 4, OLS_KALMAN, 128),
    _pick("ols", 8, OLS_KALMAN), _pick("ols", 16, OLS_NLMS), _pick("ols", 16, OLS_KALMAN),
    _pick("ols1024", 4, OLS_NLMS), _pick("ols1024", 8, OLS_KALMAN),
    _pick("feat", 4, NLMS, 200), _pick("feat", 4, KALMAN, 200),
]

# Non-default filter parameters, chosen where the float32 oracle stays >= 10x below the bar (measured drift of the
# float32 restatement against float64 on the rows of test_filter_parameters_match_oracle: <= 6e-7 for every set, at every
# path below).  Across the sets every field a step rule reads takes a non-default value.
PARAMS = {
    NLMS: [dict(mu=0.1, delta=1.0), dict(mu=1.0, delta=0.05)],
    KALMAN: [dict(kalman_a=0.99, kalman_lambda=0.5, kalman_c0=0.05, kalman_eps=1e-4),
             dict(kalman_a=0.995, kalman_lambda=0.8, kalman_c0=3.0, kalman_eps=1e-6)],
    OLS_NLMS: [dict(pb_lambda=0.0, mu=1.0, delta=0.05), dict(pb_lambda=0.95, mu=0.2, delta=1.0)],
}
PARAMS[OLS_KALMAN] = PARAMS[KALMAN]
PARAMS_P16_NLMS = dict(mu=1.5)          # the ring kernel's NLMS step at P = 16, a large step


def _param_cases():
    cases = []
    for b in [_pick("nw1", 4, NLMS, 255), _pick("nw2", 4, NLMS, 128), _pick("nw2", 4, KALMAN, 168),
              _pick("nw4", 8, NLMS, 168), _pick("nw4", 8, KALMAN, 168), _pick("nw8", 8, NLMS), _pick("nw8", 8, KALMAN),
              _pick("nw8", 16, NLMS), _pick("nw8", 16, KALMAN), _pick("1024", 8, NLMS), _pick("1024", 8, KALMAN),
              _pick("ols", 4, OLS_NLMS, 128), _pick("ols", 4, OLS_KALMAN, 128), _pick("ols", 16, OLS_NLMS),
              _pick("ols", 16, OLS_KALMAN), _pick("ols1024", 8, OLS_NLMS), _pick("ols1024", 8, OLS_KALMAN),
              _pick("feat", 4, NLMS, 200), _pick("feat", 4, KALMAN, 200)]:
        sets = list(PARAMS[b.algo])
        if b.entry == "nw8" and b.P == 16 and b.algo == NLMS:
            sets.append(PARAMS_P16_NLMS)
        for i, s in enumerate(sets):
            cases.append(pytest.param(b, s, id=f"{_bid(b)}-set{i}"))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("b,params", _param_cases())
def test_filter_parameters_match_oracle(b, params):
    """mu, delta, kalman_a / lambda / c0 / eps and pb_lambda away from their defaults reach every copy of the
    recurrence (two utterances of 16 123 samples)"""
    far, mic, hop = _signals(b.frame, b.P, 70, 2, L_LONG)
    lens = [L_LONG] * 2
    ref = O.stage1(far, mic, _oracle_cfg(b, **params), erle_skip=SKIP * hop)
    _check(b, _run(b, far, mic, **params), ref, lens)


TONE_BINS = {512: (0, 1, 127, 128, 129, 255, 256), 1024: (0, 1, 255, 256, 257, 511, 512)}


def tone_rows(frame, L=L_LONG):
    """one row per bin k of TONE_BINS[frame]: far = 0.5 cos(2 pi k n / N + phi) at the bin centre (phi = 0 at DC and
    Nyquist, where the signal is real-valued in the bin, else 0.3 + 0.1 k), mic = 0.6 x far delayed by 37 samples plus
    white noise 60 dB below that echo"""
    n = np.arange(L)
    rng = np.random.default_rng(frame)
    far, mic = [], []
    for k in TONE_BINS[frame]:
        phi = 0.0 if k in (0, frame // 2) else 0.3 + 0.1 * k
        x = 0.5 * np.cos(2 * np.pi * k * n / frame + phi)
        echo = 0.6 * np.concatenate([np.zeros(37), x[:-37]])
        noise = rng.standard_normal(L) * np.sqrt(np.mean(echo ** 2)) * 1e-3
        far.append(x)
        mic.append(echo + noise)
    return np.array(far, dtype=np.float32), np.array(mic, dtype=np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("b", PATHS, ids=_bid)
def test_tones_at_the_special_bins_match_oracle(b):
    """DC and Nyquist (packed into one complex value), the self-mirrored bin N / 4 (serial pass, or one chunk ahead on
    the ring kernel) and their neighbours, each carrying the whole far end"""
    far, mic = tone_rows(b.frame)
    ref = O.stage1(far, mic, _oracle_cfg(b), erle_skip=SKIP * _hop(b))
    _check(b, _run(b, far, mic), ref, [far.shape[1]] * far.shape[0])


LEVELS = (1.0, 1e-2, 1e-3, 3e-5)       # 3e-5 of a 0.5-peak far end is about 1 LSB of 16-bit PCM


def level_rows(frame, P, L=L_LONG):
    from acoustic_echo_cancellation_b200 import synth
    u = synth.make_utterance(9, L, sample_rate=16000 * frame // 512, rir_len=min(P * frame // 2, 4096))
    s = np.array(LEVELS, dtype=np.float32)[:, None]
    return (u["far"][None] * s).astype(np.float32), (u["mic"][None] * s).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("b", PATHS, ids=_bid)
def test_quiet_signals_match_oracle_relative_to_their_level(b):
    """one utterance at 1, 1e-2, 1e-3 and 3e-5 of its level, one level per row: each row within 1e-4 x max|mic| of the
    oracle (at 3e-5 the absolute bar alone would pass a kernel that wrote zeros), and within the absolute bar"""
    far, mic = level_rows(b.frame, b.P)
    ref = O.stage1(far, mic, _oracle_cfg(b), erle_skip=SKIP * _hop(b))
    out = _run(b, far, mic)
    lens = [far.shape[1]] * far.shape[0]
    _check(b, out, ref, lens)
    _check(b, out, ref, lens, tol=TOL_ERR * np.abs(mic).max(axis=1))
