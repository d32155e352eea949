"""A/B of the config-3 (non-stationary, n_fft 2048, 64 ch x 10 min @ 48 kHz) kernel variants on one B200: step time, stage
times from the library, and agreement of the outputs.   python scripts/ab_config3.py [flags ...]
path_flags: 0 default | 128 tap-loop smoothing (k_smooth_stream) | 64 follower stores its forward sweep"""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import synth_device, SR, C_PER_GPU  # noqa: E402
from noisereduce_b200.device import DeviceGate  # noqa: E402

flags = [a for a in sys.argv[1:]] or ["0", "128", "64"]     # an argument "v:NAME" times libb200gate_NAME.so (scripts/build_variant.py) with path_flags 0
dev = torch.device("cuda", 0)
n = 10 * 60 * SR
x = synth_device(torch, C_PER_GPU, n, 0, dev)
out = torch.empty_like(x)
base = None
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for arg in flags:
    lib = None
    f = 0
    if arg.startswith("v:"):
        from noisereduce_b200 import _cabi
        lib = _cabi.GateLibrary(os.path.join(ROOT, "noisereduce_b200", f"libb200gate_{arg[2:]}.so"))
    else:
        f = int(arg)
    dg = DeviceGate(sr=SR, stationary=False, n_fft=2048, workspace_limit_bytes=72e9, path_flags=f, lib=lib)
    for _ in range(2):
        dg.run(x, out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    K = 4
    for _ in range(K):
        dg.run(x, out)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / K
    s = dg.gate.stats()
    sub = out[:, : 3 * 600000].clone()
    if base is None:
        base = sub
    print(json.dumps({"variant": arg, "path_flags": f, "ms_per_step": round(ms, 2), "gsamples_per_s": round(C_PER_GPU * n / ms / 1e6, 2),
                      "analysis_ms": round(s["k1_ms"], 2), "follower+smoothing_ms": round(s["smooth_ms"], 2),
                      "synthesis_ms": round(s["k2_ms"], 2), "launches": s["kernel_launches"],
                      "max_abs_diff_vs_first": float((sub - base).abs().max().item()),
                      "out_absmax": float(sub.abs().max().item())}), flush=True)
    del dg
