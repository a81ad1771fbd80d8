"""Streaming stage 1 (aec_stage1_run_stream) against the one-shot overlap-save kernel, on the current GPU.

(a) 1024 utterances x 10 s, algos 2 and 3 at P = 4, 8 and 16: one stream call per utterance (the whole utterance as
    one chunk) against stage1_aec, the two alternated (inputs of 1.3 GB: far beyond L2).
(b) the same audio cut into chunks of 1, 2, 5, 20 and 625 blocks (256 samples) for 1024 and 4096 streams at P = 4:
    device time per call, audio seconds per second, and the state bytes one call moves (load + store) against its
    signal bytes (far, mic in, err out).  The timed calls rotate over R independent sets of states and buffers, R chosen
    so that the sets together hold at least 4x the L2 size: every call's state and signal come from HBM, not from what
    the previous call left in L2.  Each row is timed three ways:
      direct  -- the calls launched from Python one after another (ctypes + the C entry's host side per call);
      graph   -- the same rotation captured once in a CUDA graph and replayed: no host work between the kernels, so
                 direct > graph means the device waited on the host;
      zero    -- graph-replayed calls with 0 blocks per row: launch, state read of the prologue, nothing else (the fixed
                 cost of a call);
    plus l2 -- direct calls on ONE set (what a server re-feeding the same slots sees when its batch fits L2).
    The byte rate of the graph time is set against the device-to-device copy rate measured in the same run (1 GiB
    tensors: read + write bytes per second), the practical HBM ceiling.
Device events around many launches after a warm-up; the card's name and power limit are read in the same run.  Writes
profiles/r3_stream_bench.json (or --out).

    python tools/stream_bench.py [--reps 20] [--out profiles/r3_stream_bench.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import acoustic_echo_cancellation_b200 as A  # noqa: E402
from acoustic_echo_cancellation_b200 import _lib, synth  # noqa: E402

H, SR, L = 256, 16000, 160000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().split("\n")[torch.cuda.current_device()]
    name, plim = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit": plim}


def audio(B):
    d = synth.make_batch(0, 16, L, sample_rate=SR, rir_len=1024)
    idx = torch.arange(B) % 16
    return torch.from_numpy(d["far"]).cuda()[idx].contiguous(), torch.from_numpy(d["mic"]).cuda()[idx].contiguous()


def timed(fn, reps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def stream_call(s, far, mic, err, n):
    lib, c = _lib.load(), s._c
    B, W = far.shape

    def go():
        stream = int(torch.cuda.current_stream().cuda_stream)           # (the capture stream inside torch.cuda.graph)
        _lib.check(lib.aec_stage1_run_stream(far.data_ptr(), mic.data_ptr(), err.data_ptr(), None, None, n.data_ptr(),
                                             B, W, W, W, C.byref(c), s.state.data_ptr(), s.state_stride, stream),
                   "aec_stage1_run_stream")
    return go


def graph_of(calls, per_graph):
    """a CUDA graph of `per_graph` calls cycling over `calls`, and a function that replays it"""
    for fn in calls:                      # first launches (kernel attributes) outside the capture
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, capture_error_mode="relaxed"):
        for i in range(per_graph):
            calls[i % len(calls)]()
    return g.replay


def copy_rate():
    """device-to-device copy of 1 GiB: (read + write bytes) / s, best of 5"""
    a = torch.empty(1 << 28, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    best = min(timed(lambda: b.copy_(a), 10) for _ in range(5))
    return 2 * a.numel() * 4 / (best * 1e-3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_stream_bench.json"))
    args = ap.parse_args()
    props = torch.cuda.get_device_properties(torch.cuda.current_device())
    l2 = int(getattr(props, "L2_cache_size", 126 << 20))
    res = {"card": card(), "l2_bytes": l2, "copy_bytes_per_s": copy_rate(),
           "audio": "synth.make_batch(0, 16, 10 s) tiled over the rows, 16 kHz", "a": [], "b": []}
    print(json.dumps({k: res[k] for k in ("card", "l2_bytes", "copy_bytes_per_s")}), flush=True)
    far, mic = audio(4096)
    # (a) one stream call per utterance against the one-shot kernel, alternated
    for P in (4, 8, 16):
        for algo in (2, 3):
            cfg = A.Stage1Config(partitions=P, algo=algo)
            f, m = far[:1024], mic[:1024]
            out = torch.empty_like(f)
            s = A.Stage1Stream(1024, cfg)
            n = torch.full((1024,), L, dtype=torch.int64, device="cuda")
            one = lambda: A.stage1_aec(f, m, cfg, out=out)      # noqa: E731
            st = stream_call(s, f, m, out, n)
            t1, t2 = [], []
            for _ in range(3):
                t1.append(timed(one, args.reps))
                t2.append(timed(st, args.reps))
            row = {"algo": algo, "P": P, "B": 1024, "seconds": 10, "one_shot_ms": min(t1), "stream_ms": min(t2),
                   "stream_over_one_shot": min(t2) / min(t1), "state_bytes_per_utterance_io": 2 * s.state_bytes,
                   "signal_bytes_per_utterance": 3 * 4 * L}
            res["a"].append(row)
            print(json.dumps(row), flush=True)
            del s, out
    # (b) chunk sizes, rotating over sets that together exceed the L2 four times
    for B in (1024, 4096):
        for algo in (2, 3):
            cfg = A.Stage1Config(partitions=4, algo=algo)
            for blocks in (1, 2, 5, 20, 625):
                W = blocks * H
                sig = 3 * 4 * W * B
                probe = A.Stage1Stream(1, cfg)
                stb = 2 * probe.state_bytes * B
                footprint = B * probe.state_stride + sig
                R = max(1, -(-4 * l2 // footprint))
                sets, zeros = [], []
                n = torch.full((B,), W, dtype=torch.int64, device="cuda")
                n0 = torch.zeros((B,), dtype=torch.int64, device="cuda")
                for r in range(R):
                    off = (r * W) % (L - W + 1) if R > 1 else 0
                    f, m = far[:B, off:off + W].contiguous(), mic[:B, off:off + W].contiguous()
                    s, err = A.Stage1Stream(B, cfg), torch.empty((B, W), dtype=torch.float32, device="cuda")
                    sets.append(stream_call(s, f, m, err, n))
                    zeros.append(stream_call(s, f, m, err, n0))
                torch.cuda.synchronize()
                calls = max(R, 20 if blocks >= 20 else 200)
                reps = max(1, calls // R)

                def direct():
                    for fn in sets:
                        fn()
                ms_direct = timed(direct, reps) / R
                ms_graph = timed(graph_of(sets, calls), 3) / calls
                ms_zero = timed(graph_of(zeros, calls), 3) / calls
                ms_l2 = timed(sets[0], calls)
                rate = (stb + sig) / (ms_graph * 1e-3)
                row = {"B": B, "algo": algo, "P": 4, "chunk_blocks": blocks, "sets_rotated": R,
                       "bytes_rotated": R * footprint, "ms_per_call_direct": ms_direct, "ms_per_call_graph": ms_graph,
                       "ms_per_call_zero_blocks_graph": ms_zero, "ms_per_call_l2_resident_direct": ms_l2,
                       "audio_s_per_s": B * W / SR / (ms_graph * 1e-3), "state_bytes_per_call": stb,
                       "signal_bytes_per_call": sig, "state_over_signal": stb / sig,
                       "bytes_per_s_state_plus_signal_graph": rate, "of_copy_rate": rate / res["copy_bytes_per_s"]}
                res["b"].append(row)
                print(json.dumps(row), flush=True)
                del sets, zeros
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
