"""Per-launch time of the transition block (x <- x + FeedForward(x), d = 256, hidden = 1024) at the C2 pair and MSA shapes:
the fused kernel (ff_tc_kernel, one launch) against the two-launch path (AF2_FF_FUSED=0), CUDA events around 50 calls after
10 warm-up calls.  The fp32 stream (67 / 34 MB) fits the 126 MB L2, so the numbers are warm-L2 times, as inside the trunk.
Prints one JSON line per (shape, path) with the tensor floor at the 1429 TFLOP/s sustained bf16 rate of MEASURED_PEAKS.json."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import alphafold2_b200 as A  # noqa: E402
from alphafold2_b200 import _lib  # noqa: E402

PEAK_TFLOPS = 1429.0
lib = _lib.load()
torch.manual_seed(0)
ff = A.FeedForward(dim=256)
for p in ff.parameters():
    torch.nn.init.normal_(p, std=0.05)
ff = ff.cuda().eval()
props = torch.cuda.get_device_properties(0)
for name, T in (("pair", 65536), ("msa", 32768)):
    x = torch.randn(T, 256, device="cuda")
    flops = 2.0 * T * 256 * 1024 * 3
    for fused in (1, 0):
        lib.af2_set_ff_fused(fused)
        for _ in range(10):
            ff.add_to_(x)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 50
        a.record()
        for _ in range(n):
            ff.add_to_(x)
        b.record()
        torch.cuda.synchronize()
        us = a.elapsed_time(b) * 1e3 / n
        print(json.dumps(dict(shape=name, T=T, path="fused" if fused else "two_launch", us_per_call=round(us, 2),
                              tflops=round(flops / us * 1e-6, 1), tensor_floor_us=round(flops / (PEAK_TFLOPS * 1e6), 1),
                              gpu=props.name)))
lib.af2_set_ff_fused(1)
