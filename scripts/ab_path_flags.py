"""A/B of path_flags variants on config 2 (device-resident): step time, per-kernel times, and bit-equality of the outputs.

    python scripts/ab_path_flags.py 0 16       # default (dual kernels) vs one unit per warp
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import synth_device, SR, C_PER_GPU  # noqa: E402
from noisereduce_b200.device import DeviceGate  # noqa: E402

flags = [int(a) for a in sys.argv[1:]] or [0, 16]
dev = torch.device("cuda", 0)
n = 10 * 60 * SR
x = synth_device(torch, C_PER_GPU, n, 0, dev)
outs = {}
for rep in range(2):                                   # interleaved repeats: clocks / thermal drift show up as disagreement
    for f in flags:
        dg = DeviceGate(sr=SR, stationary=True, n_fft=1024, hop_length=256, workspace_limit_bytes=64e9, path_flags=f)
        dg.noise_stats(x)
        out = torch.empty_like(x)
        for _ in range(3):
            dg.run(x, out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            dg.run(x, out)
        e1.record()
        torch.cuda.synchronize()
        s = dg.gate.stats()
        print(f"rep {rep} path_flags={f}: step {e0.elapsed_time(e1) / 5:.2f} ms  k1 {s['k1_ms']:.2f}  smooth {s['smooth_ms']:.2f}  "
              f"k2 {s['k2_ms']:.2f}", flush=True)
        if rep == 0:
            outs[f] = out[:4].clone()
        del dg
base = outs[flags[0]]
for f in flags[1:]:
    print(f"path_flags={f} output bit-equal to path_flags={flags[0]}: {bool(torch.equal(base, outs[f]))}")
