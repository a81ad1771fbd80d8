"""Launch time of the overlap-save kernel against the number of resident utterances per SM (1 .. 9 x 148).
    python tools/ols_stair.py [algo] [P] [variant] [counts]
variant: 0 (default build) or the full 1000 * warps + register cap, e.g. 2168 at P <= 4 (2 warps), 4128 at P = 8,
8128 at P = 16; a bare register cap such as 168 is refused."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import acoustic_echo_cancellation_b200 as A  # noqa: E402

algo = int(sys.argv[1]) if len(sys.argv) > 1 else 2
P = int(sys.argv[2]) if len(sys.argv) > 2 else 4
variant = int(sys.argv[3]) if len(sys.argv) > 3 else 0
counts = [int(x) for x in sys.argv[4].split(',')] if len(sys.argv) > 4 else list(range(1, 10))
L = 160000
g = torch.Generator(device="cuda").manual_seed(1)
Bmax = 148 * 9
far = 0.1 * torch.randn(Bmax, L, device="cuda", generator=g)
mic = 0.5 * torch.roll(far, 37, dims=1) + 0.001 * torch.randn(Bmax, L, device="cuda", generator=g)
out = torch.empty_like(far)
cfg = A.Stage1Config(partitions=P, algo=algo, erle_skip_hops=125, variant=variant)
for n in counts:
    B = 148 * n
    for _ in range(2):
        A.stage1_aec(far[:B], mic[:B], cfg, out=out[:B])
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(4):
        A.stage1_aec(far[:B], mic[:B], cfg, out=out[:B])
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / 4
    print(f"algo {algo} P {P} variant {variant}: {n} per SM (B={B}): {ms:.3f} ms  {ms * 1.965e6 / 625:.0f} cycles/block  {B * 10 / ms / 1e3:.2f} M audio-s/s", flush=True)
