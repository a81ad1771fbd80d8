"""Streaming Stage 2 (aec_stage2_run_stream) and the streamed two-stage chain, on the current GPU.

(a) chunk sizes: 1024, 4096, 16384 and 65536 streams x 1, 2, 5 and 20 hops (256 samples) per call.  The timed calls
    rotate over R independent sets of states and buffers, R chosen so that the sets together hold at least 4x the L2
    size: every call's state and signal come from HBM.  Each row is timed three ways:
      direct -- the calls launched from Python one after another (ctypes + the C entry's host side per call);
      graph  -- the same rotation captured once in a CUDA graph and replayed (no host work between the kernels);
      zero   -- graph-replayed calls with 0 hops per row: launch, weight staging, the zero fill of the output, nothing
                else (the fixed cost of a call).
    The state bytes (load + store) and signal bytes (mic, ref in, out) per call, and their rate over the graph time
    against the device-to-device copy rate measured in the same run.
(b) 625 hops (10 s at 16 kHz in one call) for 1024 and 4096 streams against the one-shot
    LittleNetInference(in_norm=False) on the same batch, the two alternated.
(c) the chain: aec_stage1_run_stream (algo 2, P = 4) then aec_stage2_run_stream on (its error, the far end), at 1 and 5
    hops for the same stream counts, graph-replayed and direct; and AecStream.process (the Python class, with its
    per-row bookkeeping) called directly.
(d) real time: the largest measured stream count whose 1-hop call (graph-replayed) fits the 16 ms of a hop at 16 kHz,
    for Stage 2 alone and for the chain.  Stream counts between or beyond the measured ones are not extrapolated.
Device events around many launches after a warm-up; the card's name and power limit are read in the same run.  Writes
profiles/r3_stage2_stream_bench.json (or --out).

    python tools/stage2_stream_bench.py [--reps 20] [--out profiles/r3_stage2_stream_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import acoustic_echo_cancellation_b200 as A  # noqa: E402
from acoustic_echo_cancellation_b200 import _lib  # noqa: E402
from stream_bench import card, copy_rate, graph_of, stream_call, timed  # noqa: E402

H, SR = 256, 16000
HOP_MS = 1e3 * H / SR
STREAMS = (1024, 4096, 16384, 65536)


def weights():
    g = np.load(os.path.join(ROOT, "tests", "golden", "reference_stage2.npz"))
    return {k[2:]: g[k] for k in g.files if k.startswith("w_")}, g["erb"]


def s2_call(s2, state, mic, ref, out, n):
    """one aec_stage2_run_stream call of Stage2Stream s2's weights on the given state and buffers"""
    lib = _lib.load()
    B, W = mic.shape

    def go():
        stream = int(torch.cuda.current_stream().cuda_stream)
        _lib.check(lib.aec_stage2_run_stream(mic.data_ptr(), ref.data_ptr(), s2.erb.data_ptr(), C.byref(s2._cw),
                                             out.data_ptr(), n.data_ptr(), B, W, W, W, state.data_ptr(),
                                             s2.state_stride, 32, stream), "aec_stage2_run_stream")
    return go


def rotate(footprint, l2):
    return max(1, -(-4 * l2 // footprint))


def time_three(sets, zeros, calls):
    R = len(sets)

    def direct():
        for fn in sets:
            fn()
    ms_direct = timed(direct, max(1, calls // R)) / R
    ms_graph = timed(graph_of(sets, calls), 3) / calls
    ms_zero = timed(graph_of(zeros, calls), 3) / calls if zeros else None
    return ms_direct, ms_graph, ms_zero


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_stage2_stream_bench.json"))
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(torch.cuda.current_device())
    l2 = int(getattr(props, "L2_cache_size", 126 << 20))
    res = {"card": card(), "l2_bytes": l2, "sm_count": props.multi_processor_count, "copy_bytes_per_s": copy_rate(),
           "signals": "white noise, 0.1 rms; weights and bank of tests/golden/reference_stage2.npz", "hop_ms": HOP_MS,
           "a": [], "b": [], "c": []}
    print(json.dumps({k: res[k] for k in ("card", "l2_bytes", "copy_bytes_per_s")}), flush=True)
    w, erb = weights()
    g = torch.Generator(device="cuda").manual_seed(0)
    probe = A.Stage2Stream(1, w, erb)
    sb = probe.state_stride
    # (a) Stage 2 alone, chunk sizes
    for B in STREAMS:
        for hops in (1, 2, 5, 20):
            W = hops * H
            sig = 3 * 4 * W * B
            stb = 2 * probe.state_bytes * B
            R = rotate(B * sb + sig, l2)
            n = torch.full((B,), W, dtype=torch.int64, device="cuda")
            n0 = torch.zeros((B,), dtype=torch.int64, device="cuda")
            sets, zeros = [], []
            for _ in range(R):
                st = torch.zeros((B, sb), dtype=torch.uint8, device="cuda")
                m = 0.1 * torch.randn((B, W), device="cuda", generator=g)
                r = 0.1 * torch.randn((B, W), device="cuda", generator=g)
                out = torch.empty((B, W), device="cuda")
                sets.append(s2_call(probe, st, m, r, out, n))
                zeros.append(s2_call(probe, st, m, r, out, n0))
            calls = max(R, 20 if hops >= 20 or B >= 16384 else 100)
            ms_direct, ms_graph, ms_zero = time_three(sets, zeros, calls)
            rate = (stb + sig) / (ms_graph * 1e-3)
            row = {"streams": B, "hops_per_call": hops, "sets_rotated": R, "ms_per_call_direct": ms_direct,
                   "ms_per_call_graph": ms_graph, "ms_per_call_zero_hops_graph": ms_zero,
                   "us_per_stream_hop_graph": 1e3 * ms_graph / (B * hops),
                   "audio_s_per_s": B * W / SR / (ms_graph * 1e-3), "state_bytes_per_call": stb,
                   "signal_bytes_per_call": sig, "bytes_per_s_state_plus_signal_graph": rate,
                   "of_copy_rate": rate / res["copy_bytes_per_s"], "fits_hop": ms_graph <= HOP_MS}
            res["a"].append(row)
            print(json.dumps(row), flush=True)
            del sets, zeros
            torch.cuda.empty_cache()
    # (b) 10 s in one call against the one-shot path
    net = A.LittleNetInference(w, erb)
    for B in (1024, 4096):
        W = 625 * H
        m = 0.1 * torch.randn((B, W), device="cuda", generator=g)
        r = 0.1 * torch.randn((B, W), device="cuda", generator=g)
        st = torch.zeros((B, sb), dtype=torch.uint8, device="cuda")
        out = torch.empty((B, W), device="cuda")
        n = torch.full((B,), W, dtype=torch.int64, device="cuda")
        stream = s2_call(probe, st, m, r, out, n)
        one = lambda: net(m, r, in_norm=False)      # noqa: E731
        t1, t2 = [], []
        for _ in range(3):
            t1.append(timed(one, max(2, args.reps // 4)))
            t2.append(timed(stream, max(2, args.reps // 4)))
        row = {"streams": B, "hops_per_call": 625, "one_shot_ms": min(t1), "stream_ms": min(t2),
               "stream_over_one_shot": min(t2) / min(t1), "audio_s_per_s_stream": B * 10 / (min(t2) * 1e-3)}
        res["b"].append(row)
        print(json.dumps(row), flush=True)
        del m, r, st, out
        torch.cuda.empty_cache()
    # (c) the chain
    cfg = A.Stage1Config(partitions=4, algo=A.ALGO_PBFDAF)
    for B in STREAMS:
        for hops in (1, 5):
            W = hops * H
            s1p = A.Stage1Stream(1, cfg)
            foot = B * (s1p.state_stride + sb) + 5 * 4 * W * B
            R = rotate(foot, l2)
            n = torch.full((B,), W, dtype=torch.int64, device="cuda")
            sets, objs = [], []
            for _ in range(R):
                s1 = A.Stage1Stream(B, cfg)
                st2 = torch.zeros((B, sb), dtype=torch.uint8, device="cuda")
                far = 0.1 * torch.randn((B, W), device="cuda", generator=g)
                mic = 0.1 * torch.randn((B, W), device="cuda", generator=g)
                err = torch.empty((B, W), device="cuda")
                out = torch.empty((B, W), device="cuda")
                a, b = stream_call(s1, far, mic, err, n), s2_call(probe, st2, err, far, out, n)
                sets.append(lambda a=a, b=b: (a(), b()))
                objs.append(s1)
            calls = max(R, 100 if B < 16384 else 20)
            ms_direct, ms_graph, _ = time_three(sets, [], calls)
            del sets, objs
            torch.cuda.empty_cache()
            # the Python class, direct calls (its gathers and bookkeeping included), rotating as above
            streams = [A.AecStream(B, cfg, w, erb) for _ in range(R)]
            far = 0.1 * torch.randn((B, W), device="cuda", generator=g)
            mic = 0.1 * torch.randn((B, W), device="cuda", generator=g)

            def cls():
                for s in streams:
                    s.process(far, mic)
            ms_class = timed(cls, max(1, calls // R)) / R
            row = {"streams": B, "hops_per_call": hops, "stage1": "algo 2, P = 4", "sets_rotated": R,
                   "ms_per_call_graph": ms_graph, "ms_per_call_direct": ms_direct,
                   "ms_per_call_aec_stream_class": ms_class, "fits_hop": ms_graph <= HOP_MS}
            res["c"].append(row)
            print(json.dumps(row), flush=True)
            del streams
            torch.cuda.empty_cache()

    def realtime(rows):
        ok = [r["streams"] for r in rows if r["hops_per_call"] == 1 and r["ms_per_call_graph"] <= HOP_MS]
        return max(ok) if ok else 0
    res["realtime_streams_measured"] = {"stage2": realtime(res["a"]), "chain": realtime(res["c"]),
                                        "rule": "largest measured stream count whose 1-hop call (graph) <= 16 ms"}
    print(json.dumps(res["realtime_streams_measured"]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
