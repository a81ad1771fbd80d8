"""Device time of the far-end delay estimator and the far-end shift next to the stage-1 kernels on the same batch, and
the PCM16 host pipeline with and without alignment.

    python tools/delay_bench.py [--batch 1024] [--seconds 10] [--reps 10] [--out result.json]

Batch: B utterances of 10 s at 16 kHz (2 x 655 MB at B = 1024, far above the 126 MB L2, so every timed pass reads
HBM).  The signals are seeded torch noise with a per-row bulk delay: the kernels' work does not depend on the values.
Device times are CUDA events around `reps` back-to-back launches after one warm-up launch of every shape.  FLOP and
byte counts are computed from the shapes (the algorithm's, not measured traffic):
    estimator, per utterance of n samples and D = max_delay: ceil(n / D) blocks x (two D-point complex FFTs,
        5 D log2 D flops each, + the two real splits and the cross-spectrum MAC, 28 D) + one inverse FFT and its split;
        bytes: far + mic read once (8 n) + the three outputs
    align: 4 n read + 4 n written
The card's name and power limit are read in the same run (nvidia-smi query) and stored with the numbers."""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import acoustic_echo_cancellation_b200 as A  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in q[torch.cuda.current_device()].split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:          # the name still comes from torch
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unknown ({e})"}


def time_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def estimator_counts(B, n, D):
    blocks = math.ceil(n / D)
    lg = math.log2(D)
    flops = B * (blocks * (2 * 5 * D * lg + 28 * D) + 5 * D * lg + 20 * D)
    return flops, B * (8 * n + 12)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1024)
    ap.add_argument("--seconds", type=float, default=10.0)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "delay_bench measures on the GPU"
    B, L = a.batch, int(a.seconds * 16000)
    g = torch.Generator(device="cuda").manual_seed(0)
    far = 0.1 * torch.randn(B, L, device="cuda", generator=g)
    d = torch.randint(0, 4000, (B,), device="cuda", generator=g)
    idx = (torch.arange(L, device="cuda")[None] - d[:, None])
    mic = torch.where(idx >= 0, far.gather(1, idx.clamp(min=0)), torch.zeros((), device="cuda"))
    mic = 0.5 * mic + 0.01 * torch.randn(B, L, device="cuda", generator=g)
    res = {"card": card(), "batch": B, "samples": L, "audio_s": B * a.seconds, "rows": []}

    def row(name, ms, flops=None, nbytes=None, **kw):
        r = {"what": name, "ms": round(ms, 4), **kw}
        if flops:
            r["gflop"] = round(flops / 1e9, 2)
            r["tflop_s"] = round(flops / (ms * 1e-3) / 1e12, 2)
        if nbytes:
            r["gbyte"] = round(nbytes / 1e9, 3)
            r["tbyte_s"] = round(nbytes / (ms * 1e-3) / 1e12, 3)
        res["rows"].append(r)
        print(json.dumps(r), flush=True)

    shift = None
    for D in (8192, 2048):
        cfg = A.DelayConfig(max_delay=D)
        ms = time_ms(lambda: A.estimate_delay(far, mic, cfg), a.reps)
        fl, by = estimator_counts(B, L, D)
        _, s, _ = A.estimate_delay(far, mic, cfg)
        torch.cuda.synchronize()
        found = float((s.long() == (d - cfg.margin).clamp(min=0)).float().mean())
        row(f"estimate D={D}", ms, fl, by, rows_with_the_planted_shift=found)
        if shift is None:
            shift = s
    out = torch.empty_like(far)
    row("align", time_ms(lambda: A.align_far(far, shift, out=out), a.reps), nbytes=8 * B * L)
    for algo, P in ((0, 4), (2, 4), (3, 4)):
        cfg = A.Stage1Config(partitions=P, algo=algo)
        e = torch.empty_like(far)
        row(f"stage1 algo {algo} P={P}", time_ms(lambda: A.stage1_aec(out, mic, cfg, out=e), a.reps))

    # PCM16 host pipeline, page-locked int16 in, float32 out
    fh = A.pinned_empty((B, L), np.int16, A.HOST_WRITE_COMBINED)
    mh = A.pinned_empty((B, L), np.int16, A.HOST_WRITE_COMBINED)
    fh[:] = (far.clamp(-1, 0.99) * 32768).to(torch.int16).cpu().numpy()
    mh[:] = (mic.clamp(-1, 0.99) * 32768).to(torch.int16).cpu().numpy()
    err = A.pinned_empty((B, L), np.float32)
    sh = np.zeros(B, np.int32)
    pipe = A.HostPipeline(128, L)
    cfg = A.Stage1Config(partitions=4, algo=A.ALGO_PBFDAF)
    for name, al in (("host pcm16 algo 2 P=4", None), ("host pcm16 algo 2 P=4 + align D=8192", A.DelayConfig())):
        kw = {"align": al, "shift": sh} if al else {}
        pipe.run(fh, mh, cfg, err=err, **kw)
        ts = []
        for _ in range(a.host_reps):
            t0 = time.perf_counter()
            pipe.run(fh, mh, cfg, err=err, **kw)
            ts.append(time.perf_counter() - t0)
        t = float(np.median(ts))
        row(name, 1e3 * t, audio_s_per_s=round(B * a.seconds / t, 1), runs_s=[round(x, 4) for x in ts])
    pipe.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
