#!/usr/bin/env python
"""bench.py -- audio-seconds per second of the stage-1 STFT + FDAF echo canceller on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4] [--dump-outputs DIR]
    (N > 1: launched by torchrun, one rank per GPU)

One "step" = one pass of the hot path over one batch of synthetic utterances:
  workload  BASELINE.json configs[1]: 1024 synthetic 10 s utterances per GPU, 16 kHz, frame 512 /
            hop 256, 4-partition FDAF-NLMS  (weak scaling: every rank owns its own 1024).
  value     whole-job audio-seconds processed per second, inputs resident in HBM, device-timed
            (CUDA events on the launching stream, max over ranks).
  e2e       same metric through the host-buffer C-ABI call with page-locked HOST buffers: H2D -> kernel ->
            D2H of the error signal, all inside the timed region.  Headline = the 16-bit PCM entry
            (aec_stage1_run_host_pcm16: what the wav corpus holds and what create_h5 feeds); the float32
            entry (aec_stage1_run_host) is reported beside it as `float32_variant`.
  also      (N = 1) configs[2], configs[3] and the many-wave batch, device-timed the same way, outside the
            headline's timed region.
  roofline  the fused stage-1 kernel against the MEASURED FP32 FFMA peak of this GPU (binding
            roofline, SURVEY.md 8d) with the HBM fraction (MEASURED_PEAKS.json) beside it.
  cpu_baseline  the C oracle (builder-authored port; the reference has no stage-1 filter) on the
            box's host cores over a bounded sample of the same workload.
  dump      --dump-outputs DIR writes what the headline's last timed step returned (rank 0's utterances): DIR/erle_db.npy,
            the per-utterance ERLE [B], and DIR/error_signal.npy, the error signal of a fixed seeded sample of utterances
            (dump_rows), both float32.  The inputs are seeded, so two builds can be compared output for output.
`--impl reference` times that CPU port alone (there is no reference implementation of this path).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    2: dict(name="configs[1]: 1024 x 10 s utterances/GPU, 16 kHz, frame 512 hop 256, 4-partition FDAF-NLMS",
            B=1024, L=160000, P=4, algo=0, frame=512, sr=16000),
    3: dict(name="configs[2]: 4096 x 10 s utterances/GPU, 16 kHz, frame 512 hop 256, 16-partition Kalman FDAF",
            B=4096, L=160000, P=16, algo=1, frame=512, sr=16000),
    4: dict(name="configs[3]: 1024 x 10 s utterances/GPU, 48 kHz, frame 1024 hop 512, 8-partition FDAF-NLMS",
            B=1024, L=480000, P=8, algo=0, frame=1024, sr=48000),
}


def flops_per_frame(N, P, algo):
    import math
    K = N // 2 + 1
    if algo >= 2:       # overlap-save filter: five real transforms per block (X, y, E, the two of the constraint), no windows
        common = 12.5 * N * math.log2(N) + 2 * N
    else:
        common = 7.5 * N * math.log2(N) + 5 * N
    return common + (16 * K * P + 12 * K if algo in (0, 2) else 31 * K * P + 11 * K)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms.  Samples are time-stamped on
    arrival; `summary(t0, t1)` reports the ones that fell inside the timed region [t0, t1] and, when
    the region is too short for three samples, the whole under-load window (the sampler keeps running
    over identical untimed launches after the timed region) -- and says which."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1, load0, load1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def collect(a, b):
            sm, mx, power, reasons = [], [], [], set()
            for ts, r in self.rows:
                if not (a <= ts <= b):
                    continue
                f = [x.strip() for x in r.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            return sm, mx, power, reasons

        sm, mx, power, reasons = collect(t0, t1)
        window = "timed region"
        if len(sm) < 3:
            sm, mx, power, reasons = collect(load0, load1)
            window = "timed region + identical untimed launches around it (region shorter than 3 samples)"
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(power),
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json (driver-measured copy bandwidth)"
        except Exception:
            pass
    return 6650.0, "fallback of B200_PROFILING.md (MEASURED_PEAKS.json absent)"


def make_inputs(torch, B, L, seed, P, SR=16000, hop=256, device="cuda", draws="host"):
    """SURVEY.md 8d recipe (seeded): speech-like far end, exponentially decaying random RIR of P*hop taps,
    mic = echo + noise at -40 dB.  ONE generator for both arms: the Gaussian draws come from a CPU
    torch.Generator (utterance block b0 uses seed + b0, so the first k utterances are the same whatever B is),
    the filtering runs on `device` -- the GPU for our arm, the host for `--impl reference`.  Untimed set-up."""
    far = torch.empty(B, L, device=device)
    mic = torch.empty(B, L, device=device)
    t = torch.arange(L, device=device, dtype=torch.float32) / SR
    env = 0.5 - 0.5 * torch.cos(2 * torch.pi * 4.0 * t)
    nfft = 1 << (L + P * hop).bit_length()
    lp = torch.fft.rfft(0.9 ** torch.arange(128, device=device, dtype=torch.float32), n=nfft)
    tau = P * hop / 6.9
    dec = torch.exp(-torch.arange(P * hop, device=device, dtype=torch.float32) / tau)
    step = 64 if L <= 200000 else 16
    pin = device != "cpu"
    for b0 in range(0, B, step):
        nb = min(step, B - b0)
        if draws == "device":      # side measurements only: same recipe, draws from the device generator
            g = torch.Generator(device=device).manual_seed(seed * 100003 + b0)
            dr = torch.randn(nb, 2 * L + P * hop, generator=g, device=device)
        else:
            g = torch.Generator(device="cpu").manual_seed(seed * 100003 + b0)
            dr = torch.randn(nb, 2 * L + P * hop, generator=g, pin_memory=pin).to(device, non_blocking=True)
        x = dr[:, :L]
        x = torch.fft.irfft(torch.fft.rfft(x, n=nfft) * lp, n=nfft)[:, :L] * env
        x = 0.5 * x / x.abs().amax(dim=1, keepdim=True)
        h = dr[:, 2 * L:] * dec
        h = 0.5 * h / h.norm(dim=1, keepdim=True)
        echo = torch.fft.irfft(torch.fft.rfft(x, n=nfft) * torch.fft.rfft(h, n=nfft), n=nfft)[:, :L]
        noise = dr[:, L:2 * L] * echo.pow(2).mean(dim=1, keepdim=True).sqrt() * 0.01
        far[b0:b0 + nb] = x
        mic[b0:b0 + nb] = echo + noise
    return far, mic


def workload_config(wl, world):
    """`config` of the JSON line -- identical for both arms."""
    B, L, SR, FRAME = wl["B"], wl["L"], wl["sr"], wl["frame"]
    return {"workload": wl["name"], "utterances_per_gpu": B, "samples": L, "sample_rate": SR,
            "frame": FRAME, "hop": FRAME // 2, "partitions": wl["P"], "algo": ("nlms", "kalman", "ols-nlms", "ols-kalman")[wl["algo"]],
            "generator": "bench.make_inputs (SURVEY 8d recipe, CPU-seeded draws, seed 1000 + rank)",
            "l2": "inputs %.1f GB/GPU per step >> 126 MB L2 (no flush needed)" % (2 * B * L * 4 / 1e9),
            "parallelism": f"utterance-sharded x{world}, metrics-only all_gather"}


DUMP_BYTES = 48 << 20       # error-signal rows of --dump-outputs: with the ERLE, well under 64 MB per dump


def dump_rows(B, L):
    """the utterances whose error signal --dump-outputs writes: a fixed seeded sample, sorted"""
    import numpy as np

    k = max(1, min(B, DUMP_BYTES // (4 * L)))
    return np.sort(np.random.default_rng(0).choice(B, size=k, replace=False))


def cpu_sample_size(cores, B):
    return int(min(512, max(32, 16 * cores), B))


def cpu_arm(np, far, mic, wl, steps, warmup):
    """C oracle (port) on all host threads; returns (audio_s_per_s, threads, ms_per_step)."""
    from oracle import aec_oracle as O
    from oracle import c_oracle as CO

    cfg = O.AecConfig(frame=wl["frame"], partitions=wl["P"], algo=wl["algo"], delta=1e-6 * wl["frame"])
    # every core this process may run on (torchrun exports OMP_NUM_THREADS=1; the explicit thread
    # count passed to the C entry overrides it)
    try:
        threads = len(os.sched_getaffinity(0))
    except AttributeError:
        threads = os.cpu_count() or 1
    out = (np.zeros_like(far), None, np.zeros(far.shape[0], dtype=np.float32))   # pre-faulted outputs
    for _ in range(warmup):
        CO.stage1(far, mic, cfg, want_echo=False, out=out, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        CO.stage1(far, mic, cfg, want_echo=False, out=out, n_threads=threads)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return far.shape[0] * far.shape[1] / wl["sr"] / dt, threads, dt * 1e3


def stft_shell_cpu(np, far, mic, frame, threads):
    """The reference's own STFT shell on the host cores (BASELINE.md 3(1), SURVEY 8d): ConvSTFT x 2 +
    ConviSTFT x 1 (Stage2_lhm/scripts/network/attention_ccrn.py:28-101) -- dense strided convolutions.  The
    reference modules themselves are timed when /root/reference is present (this container); on the GPU box it is
    not, and the same dense-conv formulation restated with torch.nn.functional is timed instead (kind "port")."""
    import torch
    import torch.nn.functional as F

    torch.set_num_threads(max(1, threads))
    hop = frame // 2
    x, y = torch.from_numpy(far), torch.from_numpy(mic)
    ref_dir = "/root/reference/Stage2_lhm/scripts"
    kind = "port"
    stft = istft = None
    if os.path.isdir(ref_dir):
        try:
            sys.path.insert(0, ref_dir)
            from network.attention_ccrn import ConvSTFT, ConviSTFT  # type: ignore

            stft = ConvSTFT(frame, hop, frame, "hann", "complex", fix=True)
            istft = ConviSTFT(frame, hop, frame, "hann", "complex", fix=True)
            kind = "reference"
        except Exception:
            stft = istft = None
        finally:
            sys.path.remove(ref_dir)
    if stft is None:
        w = torch.hann_window(frame, periodic=True, dtype=torch.float64)
        basis = torch.fft.rfft(torch.eye(frame, dtype=torch.float64))
        k = torch.cat([basis.real, basis.imag], 1).T
        kf = (k * w)[:, None, :].float()
        ki = (torch.linalg.pinv(k).T * w)[:, None, :].float()
        eye = torch.eye(frame)[:, None, :]
        wf = w.float()

        def stft(v):
            return F.conv1d(F.pad(v[:, None, :], [frame - hop, frame - hop]), kf, stride=hop)

        def istft(sp):
            o = F.conv_transpose1d(sp, ki, stride=hop)
            tt = (wf[None, :, None] ** 2).repeat(1, 1, sp.size(-1))
            coff = F.conv_transpose1d(tt, eye, stride=hop)
            return (o / (coff + 1e-8))[..., frame - hop:-(frame - hop)]

    with torch.no_grad():
        istft(stft(x[:2]) - stft(y[:2]))                      # warm-up
        t0 = time.perf_counter()
        istft(stft(y) - stft(x))
        dt = time.perf_counter() - t0
    return {"kind": kind, "seconds": dt, "utterances": int(far.shape[0]), "threads": threads,
            "what": "ConvSTFT x 2 + ConviSTFT x 1 only (no filter): attention_ccrn.py:28-101"}


def run_reference(args, wl):
    """`--impl reference`: the CPU arm.  The reference repository has no implementation of this
    path (no FDAF at all), so the arm is the builder-authored C port on the host cores, on the first utterances
    of the SAME generator, seed and configuration as our arm."""
    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = cpu_sample_size(cores, wl["B"])
    torch.set_num_threads(cores)
    far, mic = make_inputs(torch, sample, wl["L"], 1000, wl["P"], wl["sr"], wl["frame"] // 2, device="cpu")
    far, mic = far.numpy(), mic.numpy()
    v, threads, ms = cpu_arm(np, far, mic, wl, args.steps, max(args.warmup, 1))
    shell = None
    try:
        n_shell = min(sample, 64)
        sh = stft_shell_cpu(np, far[:n_shell], mic[:n_shell], wl["frame"], threads)
        sh["audio_s_per_s"] = n_shell * wl["L"] / wl["sr"] / sh["seconds"]
        shell = sh
    except Exception as e:      # the shell figure is context, never the arm's value
        shell = {"unavailable": repr(e)}
    line = {
        "impl": "reference", "metric": "audio_seconds_per_second_stage1_aec", "value": v, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded: speech-like far end, random decaying RIR, -40 dB noise)",
        "config": workload_config(wl, args.gpus),
        "cpu_baseline": {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port",
                         "sample": f"first {sample} utterances x {wl['L'] / wl['sr']:.0f} s of the workload per step, C "
                                   f"oracle (oracle/csrc/aec_oracle.c, builder-authored port: the reference has no CPU "
                                   f"FDAF to time), OpenMP over utterances",
                         "reference_stft_shell": shell},
        "e2e": {"value": v, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "parity": "FDAF recurrence: parity UNPINNED (no reference implementation); STFT/iSTFT pinned by golden vectors",
    }
    print(json.dumps(line), flush=True)


def device_timed(A, torch, dist, sharding, far, mic, err, cfg, steps, world, n_total):
    """K steps of the device-resident path, CUDA events on the launching stream (whole region and per launch);
    returns (total_ms, mean_kernel_ms, launches, last erle, wall window)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    barrier()
    A.launch_count(reset=True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    wall0 = time.perf_counter()
    ev0.record()
    pending = []
    erle = None
    for i in range(steps):
        kev[i][0].record()
        erle = A.stage1_aec(far, mic, cfg, out=err, return_erle=True)[1]
        kev[i][1].record()
        if world > 1:     # metrics gather of step i runs on NCCL's stream under the kernel of step i + 1
            pending.append(sharding.gather_metrics(erle, n_total, async_op=True))
    for _, work in pending:
        if work is not None:
            work.wait()   # every step's gathered metrics are complete inside the timed region
    ev1.record()
    barrier()
    wall1 = time.perf_counter()
    launches = A.launch_count()
    total_ms = ev0.elapsed_time(ev1)
    kern_ms = sum(a.elapsed_time(b) for a, b in kev) / steps
    return total_ms, kern_ms, launches, erle, (wall0, wall1)


def roofline_of(wl, kern_ms, fp32_peak, hbm_peak, hbm_src, traffic=None):
    frames = wl["L"] // (wl["frame"] // 2) + (1 if wl["algo"] < 2 else 0)     # overlap-save: whole blocks only
    flops_launch = flops_per_frame(wl["frame"], wl["P"], wl["algo"]) * frames * wl["B"]
    bytes_launch = 3 * 4 * wl["L"] * wl["B"]
    tf = flops_launch / (kern_ms * 1e-3) / 1e12
    gbs = bytes_launch / (kern_ms * 1e-3) / 1e9
    return {"bound": "fp32", "achieved": tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": tf / fp32_peak,
            "traffic": traffic, "kernel": "aec::stage1_n%d_kernel" % wl["frame"] if wl["algo"] < 2 else
            ("aec::stage1_ols_kernel" if wl["frame"] == 512 else "aec::stage1_ols1024_kernel"),
            "kernel_ms": kern_ms,
            "flops_per_launch": flops_launch, "bytes_per_launch": bytes_launch,
            "peak_source": "FFMA probe measured live in this run (aec_bench_fp32_peak; FFMAs with constant operands -- "
                           "FFMAs with three register sources issue at 0.64 of it, profiles/r2_ffma_reuse.txt); "
                           "MEASURED_PEAKS.json carries no FP32 figure",
            "hbm": {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "peak_source": hbm_src}}


def fused_row(A, torch, wl, far, mic, err, cfg, args, fp32_peak, local):
    """stage 1 + Stage-2 front end in one launch, against the two-launch pipeline on the same inputs (device-timed)"""
    erb = torch.from_numpy(A.erb_filterbank()).float().cuda()
    steps = max(5, min(args.steps, 20))

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        A.launch_count(reset=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps, A.launch_count()

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.1)
    w0 = time.perf_counter()
    fused_ms, launches = timed(lambda: A.stage1_aec_features(far, mic, erb, cfg, out=err))
    two_ms, _ = timed(lambda: (A.stage1_aec(far, mic, cfg, out=err), A.stage2_features(err, far, erb, in_norm=False)))
    while time.perf_counter() - w0 < 0.35:
        A.stage1_aec_features(far, mic, erb, cfg, out=err)
        torch.cuda.synchronize()
    w1 = time.perf_counter()
    time.sleep(0.05)
    sampler.stop()
    _, feat = A.stage1_aec_features(far, mic, erb, cfg, out=err)
    want = A.stage2_features(err, far, erb, in_norm=False)
    B, L = far.shape
    return {"workload": wl["name"], "ms_per_step": fused_ms, "steps": steps,
            "value": B * L / wl["sr"] / (fused_ms * 1e-3), "unit": "audio-s/s",
            "two_launch_pipeline_ms": two_ms, "speedup_vs_two_launches": two_ms / fused_ms,
            "features_max_abs_diff_vs_standalone": float((feat - want).abs().max()), "features_scale": float(want.abs().max()),
            "hbm_bytes_algorithmic": {"fused": 3 * 4 * B * L + 4 * feat.numel(), "two_launches": 5 * 4 * B * L + 4 * feat.numel()},
            "gpu_launches": int(launches), "outputs_finite": bool(torch.isfinite(feat).all()),
            "clocks": sampler.summary(w0, w1, w0, w1)}


def also_rows(A, torch, sharding, args, fp32_peak, hbm_peak, hbm_src, local):
    """Outside the headline's timed region (N = 1 only): the other single-GPU configurations of BASELINE.json and
    the many-wave batch, device-timed with the same method, so that they exist in the driver's record."""
    rows = []
    extra = [dict(WORKLOADS[3]), dict(WORKLOADS[4]),
             dict(WORKLOADS[2], B=4144, name="many waves: 4144 x 10 s utterances (28 per SM), 16 kHz, 4-partition FDAF-NLMS"),
             dict(WORKLOADS[2], algo=2, name="configs[1] through the overlap-save PBFDAF (algo 2: exact linear convolution, "
                                             "alternated constraint, NLMS step; ~38 dB ERLE where the STFT-domain filter "
                                             "reaches 13)"),
             dict(WORKLOADS[2], algo=3, name="configs[1] through the overlap-save PBFDAF with the Kalman step (algo 3)"),
             dict(WORKLOADS[3], algo=3, name="configs[2] through the overlap-save PBFDAF with the Kalman step (algo 3, 16 "
                                             "partitions, eight warps per utterance)"),
             dict(WORKLOADS[4], algo=3, name="configs[3] through the overlap-save PBFDAF with the Kalman step (algo 3, frame 1024, 8 "
                                             "partitions: the double-talk configuration through the double-talk-robust filter)"),
             dict(WORKLOADS[2], feat=True, name="configs[1] with the Stage-2 feature front end fused into the kernel "
                                                "(aec_stage1_run_features: error signal + [B, T, 64] features per launch)")]
    for wl in extra:
        try:
            far, mic = make_inputs(torch, wl["B"], wl["L"], 7, wl["P"], wl["sr"], wl["frame"] // 2, device="cuda",
                                   draws="device")
            err = torch.empty_like(far)
            cfg = A.Stage1Config(frame=wl["frame"], partitions=wl["P"], algo=wl["algo"], erle_skip_hops=125)
            if wl.get("feat"):
                rows.append(fused_row(A, torch, wl, far, mic, err, cfg, args, fp32_peak, local))
                del far, mic, err
                torch.cuda.empty_cache()
                continue
            for _ in range(3):
                A.stage1_aec(far, mic, cfg, out=err, return_erle=True)
            torch.cuda.synchronize()
            sampler = ClockSampler(local)
            sampler.start()
            time.sleep(0.1)
            load0 = time.perf_counter()
            steps = max(5, min(args.steps, 20))
            total_ms, kern_ms, launches, erle, (w0, w1) = device_timed(A, torch, None, sharding, far, mic, err, cfg, steps,
                                                                      1, wl["B"])
            while time.perf_counter() - load0 < 0.35:          # keep the same load up until the sampler has >= 3 samples
                A.stage1_aec(far, mic, cfg, out=err, return_erle=True)
                torch.cuda.synchronize()
            load1 = time.perf_counter()
            time.sleep(0.05)
            sampler.stop()
            ms = total_ms / steps
            rf = roofline_of(wl, kern_ms, fp32_peak, hbm_peak, hbm_src)
            cpu_port = None
            if wl["algo"] >= 2 and wl["B"] <= 1024 and wl["frame"] == 512 and not args.no_cpu_baseline:
                import numpy as np                              # the same filter through the C port, bounded sample
                ns_ = cpu_sample_size(os.cpu_count() or 1, wl["B"])
                v_, th_, _ = cpu_arm(np, far[:ns_].cpu().numpy(), mic[:ns_].cpu().numpy(), wl, 1, 1)
                cpu_port = {"value": v_, "unit": "audio-s/s", "cores": th_, "kind": "port",
                            "sample": f"first {ns_} utterances of this row's batch, 1 timed pass, C oracle (run_group_ols)"}
            rows.append({"workload": wl["name"], "ms_per_step": ms, "steps": steps, "cpu_port": cpu_port,
                         "value": wl["B"] * wl["L"] / wl["sr"] / (ms * 1e-3), "unit": "audio-s/s",
                         "roofline": {"frac": rf["frac"], "achieved": rf["achieved"], "peak": rf["peak"], "unit": rf["unit"],
                                      "hbm_frac": rf["hbm"]["frac"], "kernel_ms": kern_ms},
                         "gpu_launches": int(launches), "erle_db_mean": float(erle.float().mean()),
                         "outputs_finite": bool(torch.isfinite(err).all()),
                         "clocks": sampler.summary(w0, w1, load0, load1)})
            del far, mic, err
            torch.cuda.empty_cache()
        except Exception as e:                                  # never lose the headline line to a side measurement
            rows.append({"workload": wl["name"], "error": repr(e)})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--algo", type=int, default=None, choices=[0, 1, 2, 3],
                    help="run the chosen config through another filter (2 / 3: the overlap-save PBFDAF); both arms")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true")
    ap.add_argument("--e2e-slots", type=int, default=0)
    ap.add_argument("--e2e-slice", type=int, default=128)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    wl = WORKLOADS[args.config]
    if args.algo is not None and args.algo != wl["algo"]:
        wl = dict(wl, algo=args.algo, name=wl["name"] + " -- run through aec_cfg.algo = %d (%s)" % (
            args.algo, ("nlms", "kalman", "ols-nlms", "ols-kalman")[args.algo]))
    if args.impl == "reference":
        return run_reference(args, wl)
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch
    import torch.distributed as dist

    import acoustic_echo_cancellation_b200 as A
    from acoustic_echo_cancellation_b200 import sharding

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: acoustic_echo_cancellation_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    numa_cpus = None
    if world > 1 and not args.no_numa_bind:
        from acoustic_echo_cancellation_b200 import hostutil
        numa_cpus = hostutil.bind_to_gpu_numa(local)     # host buffers of the e2e leg land GPU-local
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    B, L, P, algo = wl["B"], wl["L"], wl["P"], wl["algo"]
    SR, FRAME = wl["sr"], wl["frame"]
    HOP = FRAME // 2
    far, mic = make_inputs(torch, B, L, 1000 + rank, P, SR, HOP, device="cuda")
    err = torch.empty_like(far)
    cfg = A.Stage1Config(frame=FRAME, partitions=P, algo=algo, erle_skip_hops=125, variant=args.variant)
    n_total = B * world

    def step():
        _, erle = A.stage1_aec(far, mic, cfg, out=err, return_erle=True)
        if world > 1:   # the path's only collective: per-utterance metrics, never the signals
            erle = sharding.gather_metrics(erle, n_total)
        return erle

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    fp32_peak = A.fp32_peak_tflops()
    barrier()

    # ---- timed region: K steps, device-timed, inputs (1.3 GB/GPU) far larger than the 126 MB L2 ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.1)
    load0 = time.perf_counter()
    for _ in range(max(3, int(0.15 / 0.002))):      # ~0.15 s of identical launches so the sampler sees load
        A.stage1_aec(far, mic, cfg, out=err, return_erle=True)
    total_ms, kern_ms, launches, erle, (wall0, wall1) = device_timed(A, torch, dist, sharding, far, mic, err, cfg,
                                                                    args.steps, world, n_total)
    dump = None
    if args.dump_outputs and rank == 0:      # device copies now (untimed), written to DIR at the end
        dump = {"error_signal": err[torch.from_numpy(dump_rows(B, L)).cuda()], "erle_db": erle}
    wall = wall1 - wall0
    clocks = None
    if rank == 0:
        if wall < 0.3:                               # keep the GPU under the same load while sampling
            t_end = time.perf_counter() + 0.3
            while time.perf_counter() < t_end:
                A.stage1_aec(far, mic, cfg, out=err, return_erle=True)
                torch.cuda.synchronize()
        load1 = time.perf_counter()
        time.sleep(0.05)
        sampler.stop()
        clocks = sampler.summary(wall0, wall1, load0, load1)
    barrier()
    tmax = torch.tensor([total_ms, kern_ms], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms, kern_ms = float(tmax[0]), float(tmax[1])
    ms_per_step = total_ms / args.steps
    audio_s_step = n_total * L / SR
    value = audio_s_step / (ms_per_step * 1e-3)
    erle_mean = float(erle.float().mean())
    finite = bool(torch.isfinite(err).all())

    # ---- e2e: page-locked HOST buffers through the host-buffer C ABI, copies inside the timed region ----
    # headline: the 16-bit PCM entry (aec_stage1_run_host_pcm16) -- the wav files of the reference's generators hold
    # 16-bit PCM and `create_h5` feeds them to this entry as such (tests: bit-identical to the float32 entry on
    # x / 32768); the float32 entry (what a caller holding librosa.load's arrays uses) is reported beside it.
    e2e = None
    e2e_match = None
    hf = hm = None
    if not args.no_e2e:
        hf, hm, he = A.pinned_empty((B, L)), A.pinned_empty((B, L)), A.pinned_empty((B, L))
        herle = np.empty(B, dtype=np.float32)
        hf[:] = far.cpu().numpy()
        hm[:] = mic.cpu().numpy()
        sl = min(args.e2e_slice, B)
        pipe = A.HostPipeline(slice_utterances=sl, max_samples=L, device=local, slots=args.e2e_slots)
        k_e2e = max(3, min(args.steps, 10))

        he2 = A.pinned_empty((B, L))
        herle2 = np.empty(B, dtype=np.float32)

        def time_host(a, b, streaming=False, cfg=cfg):
            """K steps through the host entry.  streaming: the steps are issued back to back in the context's deferred
            mode (a call returns once its last slice is enqueued; outputs alternate between two buffers) and ONE wait
            at the end of the timed region completes them -- every copy and kernel of every step is inside the region."""
            for _ in range(2):
                pipe.run(a, b, cfg, err=he, erle=herle)
            barrier()
            t0 = time.perf_counter()
            for i in range(k_e2e):
                if streaming:
                    pipe.run(a, b, cfg, err=(he, he2)[i & 1], erle=(herle, herle2)[i & 1], wait=False)
                else:
                    pipe.run(a, b, cfg, err=he, erle=herle)     # returns when the outputs are in host memory
            if streaming:
                pipe.wait()
            barrier()
            dt = torch.tensor([(time.perf_counter() - t0) / k_e2e], device="cuda", dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            return float(dt[0])

        dt32 = time_host(hf, hm)
        e2e_match32 = bool(np.array_equal(he, err.cpu().numpy()))
        f32_variant = {"value": audio_s_step / dt32, "unit": "audio-s/s",
                       "h2d_bytes_per_step": 2 * B * L * 4, "d2h_bytes_per_step": B * L * 4 + B * 4,
                       "ms_per_step": dt32 * 1e3, "bitwise_equal_to_device_path": e2e_match32,
                       "api": "aec_stage1_run_host: float32 page-locked host memory in (H2D %.2f GB/step)" % (2 * B * L * 4 / 1e9)}
        h16f = A.pinned_empty((B, L), dtype=np.int16)
        h16m = A.pinned_empty((B, L), dtype=np.int16)
        h16f[:] = np.clip(np.rint(hf * 32768.0), -32768, 32767).astype(np.int16)
        h16m[:] = np.clip(np.rint(hm * 32768.0), -32768, 32767).astype(np.int16)
        dt16_sync = time_host(h16f, h16m)
        he16 = he.copy()
        dt16 = time_host(h16f, h16m, streaming=True)
        stream_match = bool(np.array_equal(he, he16) and np.array_equal(he2, he16))
        # the float32 entry on the de-quantised samples must give the same bits
        hf[:] = h16f.astype(np.float32) * np.float32(1.0 / 32768.0)
        hm[:] = h16m.astype(np.float32) * np.float32(1.0 / 32768.0)
        pipe.run(hf, hm, cfg, err=he, erle=herle)
        e2e_match = bool(np.array_equal(he, he16))
        hf[:] = far.cpu().numpy()
        hm[:] = mic.cpu().numpy()
        # the same end-to-end call through the overlap-save filter with the Kalman step (algo 3): the kernel is 2x the
        # time of the headline's, the step is the same -- the host link, not the filter, sets the end-to-end rate
        ols_variant = None
        if wl["frame"] == 512 and wl["P"] <= 16:
            try:
                cfg3 = A.Stage1Config(frame=wl["frame"], partitions=wl["P"], algo=3, erle_skip_hops=125)
                dt16_ols = time_host(h16f, h16m, cfg=cfg3)
                ols_variant = {"value": audio_s_step / dt16_ols, "unit": "audio-s/s", "ms_per_step": dt16_ols * 1e3,
                               "algo": "ols-kalman (aec_cfg.algo = 3), same PCM16 host entry, per call",
                               "outputs_finite": bool(np.isfinite(he).all())}
            except Exception as e:                              # never lose the headline to a side measurement
                ols_variant = {"error": repr(e)}
        e2e = {"value": audio_s_step / dt16_sync, "unit": "audio-s/s",
               "h2d_bytes_per_step": 2 * B * L * 2, "d2h_bytes_per_step": B * L * 4 + B * 4,
               "ms_per_step": dt16_sync * 1e3, "steps": k_e2e, "per_gpu": audio_s_step / dt16_sync / world,
               "api": "aec_stage1_run_host_pcm16 (HostPipeline.run): int16 PCM (the wav sample format) in page-locked host "
                      "memory -> H2D -> x/32768 on the GPU -> stage-1 kernel -> D2H of the float32 error signal + ERLE; "
                      "%d-utterance slices (ramped / tapered), %d slices in flight" % (sl, args.e2e_slots or 4),
               "mode": "per call: every step returns with its outputs in host memory",
               "bitwise_equal_to_float32_entry": e2e_match,
               "streaming_variant": {"value": audio_s_step / dt16, "unit": "audio-s/s", "ms_per_step": dt16 * 1e3,
                                     "equals_per_call": stream_match,
                                     "note": "the K steps issued back to back in the context's deferred mode "
                                             "(aec_host_ctx_set_deferred), one aec_host_ctx_wait inside the timed region"},
               "float32_variant": f32_variant, "overlap_save_kalman_variant": ols_variant}
        pipe.close()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel ----
    hbm_peak, hbm_src = measured_peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.algo is None:    # the captured traffic belongs to the config's own filter
        try:
            traffic = json.load(open(tpath)).get(f"config{args.config}")
        except Exception:
            traffic = None
    roofline = roofline_of(wl, kern_ms, fp32_peak, hbm_peak, hbm_src, traffic)

    # ---- CPU baseline: the C port on this box's cores, bounded sample of the same workload ----
    cpu = None
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = cpu_sample_size(cores, B)
        sf, sm_ = far[:sample].cpu().numpy(), mic[:sample].cpu().numpy()
        v, threads, _ = cpu_arm(np, sf, sm_, wl, 2, 1)
        cpu = {"value": v, "unit": "audio-s/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} utterances x {L / SR:.0f} s of the same workload, 2 timed passes, C oracle "
                         f"(builder-authored port: the reference has no stage-1 filter), OpenMP over utterances"}

    also = None
    if world == 1 and args.config == 2 and not args.no_also:
        del far, mic, err
        torch.cuda.empty_cache()
        also = also_rows(A, torch, sharding, args, fp32_peak, hbm_peak, hbm_src, local)

    line = {
        "metric": "audio_seconds_per_second_stage1_aec", "value": value, "unit": "audio-s/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic (seeded: speech-like far end, random decaying RIR, -40 dB noise)",
        "config": workload_config(wl, world),
        "host_cpus_rank0": (f"{len(numa_cpus)} GPU-local CPUs" if numa_cpus else "unbound"),
        "per_gpu": value / world,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "roofline": roofline,
        "roofline_hbm": {"bound": "hbm", "achieved": roofline["hbm"]["achieved"], "peak": roofline["hbm"]["peak"],
                         "unit": "GB/s", "frac": roofline["hbm"]["frac"], "traffic": traffic,
                         "note": "secondary: the binding roofline of this path is FP32 (see roofline)"},
        "cpu_baseline": cpu, "clocks": clocks, "also": also,
        "wall_s_timed_region": wall, "erle_db_mean": erle_mean, "outputs_finite": finite,
        "parity": "FDAF recurrence: parity UNPINNED (no reference implementation); STFT/iSTFT pinned by golden vectors",
    }
    if dump is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dump.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
