#!/usr/bin/env python
"""bench.py -- headline benchmark: audio samples/s denoised (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload at N=1 = BASELINE.json configs[1]: 64 ch x 10 min synthetic 48 kHz, stationary reduce_noise,
n_fft=1024 hop=256 (1.8432 G samples per step).  A step is one full pass of the hot path
(k1d_analyze -> k_rowfloor -> k_smooth -> k2d_synthesize over all 3072 (chunk, channel) units).

  value        samples/s with input and output resident in HBM (CUDA events, max over ranks)
  e2e          the same metric through the C-ABI call with HOST (pinned) buffers: H2D of the input and
               D2H of the result inside the timed region
  e2e_numpy    the same through reduce_noise() itself on a pageable numpy array (what a user of the reference calls)
  roofline     dominant kernel (k2d_synthesize: mask apply -> iSTFT): 8 algorithmic bytes per output sample / its
               CUDA-event time, against the measured HBM copy bandwidth; whole_step is the same for the whole pipeline
  parity       same-run check of the timed tensor against oracle/ on SURVEY.md section 8d's subsets
               (channels {0,31,63} x chunks {0,1,47}, thresholds of the full 64-channel clip)
  configs_extra  BASELINE configs 3 (non-stationary, n_fft 2048) and 4 (TorchGate 256 x 10 s @ 16 kHz): device-resident
               samples/s, whole-step roofline fraction, CPU legs
  cpu_baseline the reference's CPU path with n_jobs=-1 on this box's host cores on a bounded sample of the workload
               (oracle/ref_port.py: the reference's scipy.signal calls and joblib fan-out), plus n_jobs=1

--impl reference times that CPU path alone (rank 0 only under torchrun).
--dump-outputs DIR writes the waveform the last timed step computed to DIR/denoised.npy (float32; every row at a fixed,
seeded sample of column blocks when the whole output exceeds 64 MB), so that two builds can be compared on the same
seeded input.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR = 48000
C_PER_GPU = 64
N_SAMPLES = 28_800_000            # 10 min @ 48 kHz
METRIC = "audio samples/sec denoised"
UNIT = "samples/s"
ALGO_BYTES_PER_SAMPLE = 8          # float32 in + float32 out (SURVEY.md section 8d)
DUMP_BYTES = 60_000_000            # --dump-outputs: array bytes written, under 64 MB with the .npy header
DUMP_BLOCK = 4096


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_bytes():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture (profiles/k2_traffic.json)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "k2_traffic.json")))["dram_bytes_per_launch"]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = sorted(float(r[1]) for r in rows)
        out["sm_mhz"] = sm[len(sm) // 2]
        out["sm_max_mhz"] = float(rows[0][2])
        out["power_w_max"] = max(float(r[3]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, nm in enumerate(names):
            if any(r[5 + i].strip().lower().startswith("active") for r in rows):
                out["reasons"].append(nm)
        out["samples"] = len(rows)
        return out


def bind_to_gpu_numa_node(torch, local_rank):
    """Pin this process (and the pages it first-touches: pinned staging buffers) to the NUMA node its GPU hangs off."""
    try:
        bdf = subprocess.run(["nvidia-smi", "-i", str(local_rank), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip()
        bdf = bdf.lower()
        if bdf.count(":") == 2 and len(bdf.split(":")[0]) == 8:
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids)
        return {"numa_node": node, "cpus": len(ids)}
    except Exception:
        return None


def synth_device(torch, C, n, c0, device):
    """SURVEY.md section 8d synthetic signal: white noise floor + a gated tone per channel."""
    g = torch.Generator(device=device).manual_seed(1000 + c0)
    y = torch.empty((C, n), dtype=torch.float32, device=device)
    t = torch.arange(n, device=device, dtype=torch.float64) / SR
    gate = ((t % 2.0) < 0.5).to(torch.float32)
    for c in range(C):
        f = 440.0 * 2.0 ** (((c0 + c) % 24) / 12.0)
        y[c] = 0.05 * torch.randn(n, device=device, generator=g)
        y[c] += 0.25 * gate * torch.sin(2 * torch.pi * torch.remainder(t * f, 1.0)).to(torch.float32)
    return y


def synth_host(np, C, n):
    """Host-side workload of the same distribution (shifted noise per channel) for the CPU legs."""
    rng = np.random.default_rng(1000)
    base = rng.standard_normal(n + C * 997, dtype=np.float32) * np.float32(0.05)
    t = np.arange(n, dtype=np.float64) / SR
    gate = 0.25 * ((t % 2.0) < 0.5)
    y = np.empty((C, n), dtype=np.float32)
    for c in range(C):
        y[c] = base[c * 997: c * 997 + n]
        y[c] += (gate * np.sin(2 * np.pi * 440.0 * 2 ** ((c % 24) / 12) * t)).astype(np.float32)
    return y


def dump_outputs(np, torch, directory, name, y):
    """Writes the [rows, n] float32 tensor `y` as directory/name.npy: whole when it fits in DUMP_BYTES, else every row
    at a fixed set of DUMP_BLOCK-sample column blocks (seeded, sorted; the same for the same shape)."""
    rows, n = y.shape
    if rows * n * 4 > DUMP_BYTES:
        blocks = DUMP_BYTES // (rows * DUMP_BLOCK * 4)
        starts = np.sort(np.random.default_rng(0).choice(n // DUMP_BLOCK, size=blocks, replace=False)) * DUMP_BLOCK
        cols = torch.from_numpy((starts[:, None] + np.arange(DUMP_BLOCK)).reshape(-1)).to(y.device)
        y = y.index_select(1, cols)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, f"{name}.npy"), y.to(torch.float32).cpu().numpy())


def cpu_reference_run(steps, warmup, channels=16, minutes=10.0, stationary=True, n_fft=1024, with_single_job=True):
    """The reference's CPU path, n_jobs=-1 (all host cores; joblib over the chunks, base.py:206-216), on a bounded
    sample of the workload: `channels` of the 64 channels, ALL chunks of the 10-minute recording.  Channels are a
    serial loop inside each chunk job (stationary.py:86) and chunks are the parallel unit, so samples/s is
    independent of the channel count; the sample keeps the real config's chunk count (48 -> at most 48 busy workers)."""
    import numpy as np
    import scipy
    import joblib
    from oracle import ref_port
    from oracle import spectral_gate_oracle as O
    cores = os.cpu_count() or 1
    n = int(minutes * 60 * SR)
    y = synth_host(np, channels, n)
    kw = dict(stationary=stationary, n_fft=n_fft)
    if n_fft == 1024:
        kw["hop_length"] = 256
    cfg = O.GateConfig(sr=SR, **kw)

    def run(arr, jobs):
        return ref_port.reduce_noise(arr, SR, cfg, n_jobs=jobs)
    for _ in range(max(0, min(warmup, 1))):           # one warm-up spawns the loky pool (BASELINE.md section 3)
        run(y[:, : 2 * 600000 + 1], -1)
    times = []
    for _ in range(max(1, steps)):
        t0 = time.perf_counter()
        run(y, -1)
        times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    n_chunks = (n - 1) // 600000 + 1
    res = dict(value=channels * n / dt, unit=UNIT, cores=cores, kind="port", n_jobs=-1, host_cores=cores,
               busy_workers_max=min(cores, n_chunks), seconds_per_step=dt,
               sample=f"{channels} of 64 ch x all {n_chunks} chunks of 600000 samples ({channels * n / 1e6:.0f} Msamples) per step, "
                      "oracle/ref_port.py (same scipy.signal calls)"
                      f"(n_jobs=-1): joblib over chunks, channels serial inside a chunk job -> samples/s independent of the channel count",
               versions={"numpy": np.__version__, "scipy": scipy.__version__, "joblib": joblib.__version__})
    if with_single_job:
        ys = y[: min(4, channels), : 2 * 600000 + 1]
        t0 = time.perf_counter()
        run(ys, 1)
        res["n_jobs_1_value"] = ys.size / (time.perf_counter() - t0)
    return res


def torchgate_cpu_leg(rows=16):
    """Config 4 CPU leg: the reference's TorchGate restated in numpy (oracle), single thread."""
    import numpy as np
    import torch
    g = torch.Generator().manual_seed(1234)
    x = 0.05 * torch.randn((rows, 160000), generator=g)
    try:
        from oracle import torchgate_oracle as TO
        t0 = time.perf_counter()
        TO.torchgate_forward(x.numpy().astype(np.float64), sr=16000)
        dt = time.perf_counter() - t0
        return {"value": rows * 160000 / dt, "unit": UNIT, "kind": "port (numpy restatement, single thread)", "threads": 1,
                "sample": f"{rows} of 256 rows x 160000 samples"}
    except Exception as exc:
        return {"value": None, "error": repr(exc)[:160]}


def same_run_parity(np, torch, dg, x, out, n_chunks=48):
    """SURVEY.md section 8d subsets of the TIMED tensor against oracle/: channels {0,31,63} x chunks {0,1,47},
    thresholds from the full 64-channel noise clip.  Waveform rel-inf per unit; mask bits with the library's own
    thresholds (flips) and with the oracle's thresholds injected (must be 0)."""
    from oracle import spectral_gate_oracle as O
    cfg = O.GateConfig(sr=SR, stationary=True, n_fft=1024, hop_length=256)
    C, n = x.shape
    cs, pad = 600000, 30000
    clip = x[:, :cs].cpu().numpy()
    yn = O.collapse_noise(clip, cs, True)
    thresh, _, _, _ = O.stationary_threshold(yn, 1024, 1024, 256, 1.5)
    own = dg.gate.noise_threshold()
    smooth, nf, nt = O.smoothing_extents(SR, 1024, 256, 500, 50)
    filt = O.smoothing_filter(nf, nt)
    chans = [c for c in (0, 31, 63) if c < C]
    chunks = [k for k in (0, 1, n_chunks - 1) if k < n_chunks]
    ymax = float(out.abs().max().item())
    scratch = torch.empty_like(out[:2])
    refs = {}

    def compare(tag):
        worst = 0.0
        for ch in chans:
            for ck in chunks:
                o_lo, o_hi = ck * cs, min((ck + 1) * cs, n)
                i1 = ck * cs - pad
                got = out[ch, o_lo:o_hi].cpu().numpy().astype(np.float64)
                worst = max(worst, float(np.abs(got - refs[(ch, ck)][0][o_lo - i1: o_hi - i1]).max()) / max(ymax, 1e-30))
        return worst

    flips_own = flips_inj = bins = 0
    for ch in chans:
        for ck in chunks:
            i1, i2 = ck * cs - pad, (ck + 1) * cs + pad
            lo, hi = max(i1, 0), min(i2, n)
            xc = np.zeros(i2 - i1, dtype=np.float32)
            xc[lo - i1: hi - i1] = x[ch, lo:hi].cpu().numpy()
            taps = O.Taps()
            yref = O.gate_stationary_unit(xc.astype(np.float64), thresh, cfg, filt, taps)
            refs[(ch, ck)] = (yref, taps.mask0)
            bins += taps.mask0.size
    out_own = compare("own")                       # `out` still holds the timed result (library's own thresholds)
    # mask decisions: tap a 2-channel run per unit (the dual kernels pair channels), own and injected thresholds
    for inject in (False, True):
        if inject:
            dg.gate.set_noise_threshold(thresh)
        for ch in chans:
            for ck in chunks:
                c0 = ch - (ch & 1)
                dg.gate.debug_select_unit(ck, ch - c0)
                dg.run(x[c0: c0 + 2], scratch)
                d = dg.gate.debug_read()
                nb = int(np.count_nonzero(d["mask0"] != refs[(ch, ck)][1]))
                if inject:
                    flips_inj += nb
                else:
                    flips_own += nb
        dg.gate.debug_select_unit(-1, 0)
    # the whole workload once more with the reference's thresholds injected: decisions then agree bit for bit
    own_rows = out[:8].clone()                   # (8 of the 64 channels, all 48 chunks, of the own-threshold result)
    dg.run(x, out)
    torch.cuda.synchronize()
    out_inj = compare("injected")
    dfull = (out[:8] - own_rows).abs()
    full_diff = {"channels": 8, "samples": int(dfull.numel()), "samples_differing": int((dfull > 0).sum().item()),
                 "max_abs_over_ymax": float(dfull.max().item()) / max(ymax, 1e-30)}
    del own_rows, dfull
    dg.gate.set_noise_threshold(own)
    return {"out_relinf": out_inj, "out_relinf_own_thresholds": out_own,
            "mask_flips_injected_thresholds": flips_inj, "mask_flips_own_thresholds": flips_own,
            "own_vs_injected_thresholds_8ch": full_diff,
            "bins": bins, "units": len(chans) * len(chunks),
            "thresholds_max_abs_diff_db": float(np.abs(own - thresh).max()),
            "subsets": "channels {0,31,63} x chunks {0,1,47} of the timed tensor; oracle float64; thresholds of the full 64-ch clip",
            "note": "the reference transforms a float32 noise clip in float32 (scipy keeps the input precision), this library in "
                    "float64: the thresholds differ by ~1e-5 dB and a bin whose level sits inside that gap decides differently "
                    "(own-threshold flips, each a local waveform difference); with the reference's thresholds injected "
                    "(b200gate_set_noise_threshold) every decision is bit-equal and the waveform agrees to float32 rounding"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--minutes", type=float, default=10.0, help="signal length per channel (default config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip parity / configs_extra / e2e_numpy (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output to DIR/denoised.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n_gpus = max(args.gpus, world)
    config = {"workload": "64ch x 10min synthetic 48kHz stationary reduce_noise n_fft=1024 hop=256 (configs[1])"
                          + (f", x{n_gpus} GPUs: 64 channels per GPU" if n_gpus > 1 else ""),
              "channels_per_gpu": C_PER_GPU, "samples_per_channel": int(args.minutes * 60 * SR),
              "chunk_size": 600000, "padding": 30000, "l2_policy": "inputs (7.4 GB) larger than L2"}
    if n_gpus > 1:
        config["all_gather_bytes_received_per_rank"] = (n_gpus - 1) * C_PER_GPU * int(args.minutes * 60 * SR) * 4

    if args.impl == "reference":
        if rank != 0:
            return
        steps = args.steps
        r = cpu_reference_run(steps, args.warmup, channels=32, minutes=args.minutes)
        cb = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "n_jobs", "host_cores", "busy_workers_max",
                                "versions", "n_jobs_1_value") if k in r}
        line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": n_gpus,
                "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": r["seconds_per_step"] * 1e3,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "cpu_baseline": cb,
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from noisereduce_b200.device import DeviceGate

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    n = int(args.minutes * 60 * SR)
    C = C_PER_GPU

    x = synth_device(torch, C, n, rank * C, device)
    # multi-GPU transport for the path's one collective (the all-gather of the final waveform):
    #   store  kernel-issued NVLink stores (b200gate_run_sharded: k_peer_push on reserved SMs + device-side barrier)
    #   peer   copy-engine pushes into symmetric memory (round 1)
    #   nccl   all-gather kernels per channel group on a side stream
    # defaults from the measured A/B (profiles/r02_scaling.md): at N = 2 the copy engines hide the 7.4 GB push completely and
    # cost no SMs; from N = 4 on the step is bound by the NVLink port and the copy kernel (more SMs at N = 8) wins
    transport = os.environ.get("B200GATE_GATHER", "peer" if world == 2 else "store") if world > 1 else None
    reserve = int(os.environ.get("B200GATE_RESERVE_SMS", {2: "12", 4: "16"}.get(world, "32")))
    push_ctas = int(os.environ.get("B200GATE_PUSH_CTAS", str(reserve)))       # one SM-filling CTA per reserved SM
    groups = int(os.environ.get("B200GATE_GROUPS", "8"))
    ps = pg = None
    if world > 1 and transport in ("store", "peer"):
        ok = 1
        try:
            if transport == "store":
                from noisereduce_b200.parallel import PeerStore
                ps = PeerStore(world, rank, (world, C, n), torch.float32, device)
            else:
                from noisereduce_b200.parallel import PeerGather
                pg = PeerGather(world, rank, (world, C, n), torch.float32, device,
                                splits=int(os.environ.get("B200GATE_PUSH_SPLITS", "1")))
        except Exception as exc:                             # e.g. no P2P mapping in this sandbox
            ok = 0
            print(f"[bench] rank {rank}: peer-memory gather unavailable ({exc!r}); using NCCL", file=sys.stderr)
        flag = torch.tensor([ok], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            ps = pg = None
            transport = "nccl"
    out = torch.empty_like(x) if (ps is None and pg is None) else None
    reserve_sms = 0
    if world > 1:
        reserve_sms = reserve if ps is not None else (16 if pg is None else 0)
    # workspace: bits + mask numerators + cached spectra of all 3072 units (41 GB) in one batch -> one launch per kernel
    dg = DeviceGate(sr=SR, stationary=True, n_fft=1024, hop_length=256, reserve_sms=reserve_sms, workspace_limit_bytes=64e9)
    # noise statistics once (stationary.py:61-81): the reference's sequential channel mean, chained over ranks
    if world == 1:
        dg.noise_stats(x)
    else:
        from noisereduce_b200.parallel import chained_noise_stats
        chained_noise_stats(dg, x, rank, world)
    gathered = torch.empty((world * C, n), dtype=torch.float32, device=device) if (world > 1 and ps is None and pg is None) else None
    comm_stream = torch.cuda.Stream() if world > 1 else None
    acc_stats = {"k1_ms": 0.0, "smooth_ms": 0.0, "k2_ms": 0.0, "fused_ms": 0.0, "kernel_launches": 0}
    if n_gpus > 1:
        config["collective"] = {
            "store": "all-gather of the final [64*N, 28.8M] float32 waveform by kernel-issued NVLink stores (b200gate_run_sharded): "
                     "the gate kernels write a rank's rows into its slice of a symmetric-memory buffer, k_peer_push (on "
                     f"{reserve_sms} SMs the gate leaves free) stores every finished {C // groups}-channel group into all peers' buffers "
                     "while the next group is computed, one device-side epoch barrier per step; no NCCL kernels, no copy engines",
            "peer": "copy-engine pushes of every finished 8-channel group into all peers' symmetric-memory buffers; device-side barrier per step",
            "nccl": "NCCL all-gather per 8-channel group on a side stream (16 SMs reserved), overlapped with the next group's kernels",
        }[transport]
        config["gather_transport"] = {"store": "kernel-nvlink-stores", "peer": "peer-copy-engine", "nccl": "nccl"}[transport]
        config["gather_ceiling_note"] = ("weak scaling with everyone gathering everything: each rank must RECEIVE (N-1) x 7.37 GB per step "
                                         "over one NVLink port (measured peer copy 0.77 TB/s): >= 67 ms at N=8 against ~25 ms of kernels")

    def step():
        if world == 1:
            dg.run(x, out)
        elif ps is not None:
            from noisereduce_b200.parallel import sharded_run_peer_store
            sharded_run_peer_store(dg, x, ps, groups=groups, push_ctas=push_ctas)
        elif pg is not None:
            from noisereduce_b200.parallel import sharded_run_peer_push
            sharded_run_peer_push(dg, x, pg, groups=groups)
        else:
            from noisereduce_b200.parallel import sharded_run_overlapped
            sharded_run_overlapped(dg, x, out, gathered, world, comm_stream, groups=groups)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    if world > 1:
        tmax = torch.tensor([ms], device=device)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    ms_per_step = ms / args.steps
    value = world * C * n / (ms_per_step * 1e-3)
    # per-kernel CUDA-event times of the LAST run of the timed loop (the library records them around each stage); with
    # channel groups (N > 1) that is one group: scale to the step
    s_ = dg.gate.stats()
    scale = groups if world > 1 else 1
    k1, sm, k2 = s_["k1_ms"] * scale, s_["smooth_ms"] * scale, s_["k2_ms"] * scale
    launches = int(s_["kernel_launches"]) * scale * args.steps
    stats = s_
    # the gathered waveform every rank holds must be what each owner computed: compare per-rank checksums
    gather_verified = None
    if world > 1:
        full = ps.buf if ps is not None else (pg.buf if pg is not None else gathered.view(world, C, n))
        mine = full[rank].sum(dtype=torch.float64).view(1)
        owners = torch.empty(world, dtype=torch.float64, device=device)
        dist.all_gather_into_tensor(owners, mine)
        seen = torch.stack([full[r].sum(dtype=torch.float64) for r in range(world)])
        okf = torch.tensor([1.0 if bool((seen == owners).all().item()) else 0.0], device=device)
        dist.all_reduce(okf, op=dist.ReduceOp.MIN)
        gather_verified = bool(okf.item() > 0)
    ref_out = out if out is not None else (ps.buf[rank] if ps is not None else pg.buf[rank])
    if args.dump_outputs and rank == 0:
        dump_outputs(np, torch, args.dump_outputs, "denoised", ref_out if world == 1 else full.reshape(world * C, n))

    # ---- end to end through the C ABI with host buffers ----------------------------------------------
    e2e = None
    if not args.no_e2e:
        try:
            hx = torch.empty((C, n), dtype=torch.float32, pin_memory=True)
            hy = torch.empty((C, n), dtype=torch.float32, pin_memory=True)
            hx.copy_(x)
            st = torch.cuda.current_stream().cuda_stream

            def e2e_step():
                dg.gate._check(dg.gate.lib.dll.b200gate_run(dg.gate._h, hx.data_ptr(), hy.data_ptr(), 0, C, n, n, n, 0, st))

            e2e_step()
            barrier()
            ksteps = max(2, min(args.steps, 4))
            t0 = time.perf_counter()
            for _ in range(ksteps):
                e2e_step()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / ksteps
            ok = 1.0
        except Exception as exc:                      # e.g. pinned-memory limits with many ranks on one host
            dt, ok, ksteps = 0.0, 0.0, 0
            e2e_err = repr(exc)[:200]
        if world > 1:
            tt = torch.tensor([dt, ok], device=device)
            dist.all_reduce(tt[0:1], op=dist.ReduceOp.MAX)
            dist.all_reduce(tt[1:2], op=dist.ReduceOp.MIN)
            dt, ok = float(tt[0].item()), float(tt[1].item())
        if ok > 0 and dt > 0:
            e2e = {"value": world * C * n / dt, "unit": UNIT, "h2d_bytes_per_step": C * n * 4,
                   "d2h_bytes_per_step": C * n * 4, "ms_per_step": dt * 1e3, "steps": ksteps,
                   "parity_vs_device_path": float((hy.to(device) - ref_out).abs().max().item()),
                   "numa_binding": numa,
                   "note": "per-rank host buffers (pinned), slab-pipelined H2D / kernels / D2H; no collective in this leg"}
        else:
            e2e = {"value": None, "unit": UNIT, "error": locals().get("e2e_err", "failed on another rank")}
        hx = hy = None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_hbm_peak()
    k2_ms = k2
    achieved = ALGO_BYTES_PER_SAMPLE * C * n / (k2_ms * 1e-3) / 1e9 if k2_ms > 0 else None
    pipe_ach = ALGO_BYTES_PER_SAMPLE * world * C * n / (ms_per_step * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": config,
        "roofline": {"bound": "hbm", "kernel": "k2d_synthesize", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic_bytes(),
                     "peak_source": peak_src, "algorithmic_bytes_per_launch": ALGO_BYTES_PER_SAMPLE * C * n,
                     "kernel_ms": {"k1d_analyze+k_rowfloor": k1, "k_smooth": sm, "k2d_synthesize": k2_ms},
                     "whole_step": {"achieved": pipe_ach, "frac": pipe_ach / (peak * world)},
                     "traffic_note": "ncu dram bytes of one k2d_synthesize launch (cached spectra + mask numerators + waveform) -- profiles/k2_traffic.json",
                     "note": "k2d reads the 32 GB spectrum cache: its real DRAM traffic runs at ~64 % of peak, i.e. it is HBM bound on "
                             "cache bytes, not on the 8 algorithmic bytes per sample",
                     "fp32_pipe": {"source": "ncu sm__pipe_fma_cycles_active / sm__pipe_alu_cycles_active of the committed captures "
                                             "(profiles/r02_m_*_full.txt), not measured in this run",
                                   "k1d_analyze_fma": 0.424, "k2d_synthesize_fma": 0.503, "k_smooth_packed_alu": 0.597,
                                   "fma_pipe_ms_per_step": 9.4,
                                   "note": "the FP32 FFT pipeline holds the FMA pipe 9.4 ms per step whatever the memory traffic: the bound that "
                                           "binds is the FP32 pipe (42-50 % busy in the two FFT kernels), not HBM -- DESIGN.md section 6"}},
        "e2e": e2e,
        "gpu_launches": launches,
        "gather_verified": gather_verified,
        "clocks": clocks,
        "exactness": {k: stats[k] for k in ("bins_rechecked_fp64", "bins_unresolved", "rowfloor_flags", "rowfloor_ambiguous")},
    }
    if n_gpus == 1 and not args.no_extras:
        # ---- the user-facing call on a pageable numpy array ---------------------------------------------
        try:
            import noisereduce_b200 as nrb
            ynp = x.cpu().numpy()
            nrb.reduce_noise(y=ynp[:2], sr=SR, stationary=True, n_fft=1024, hop_length=256)
            calls = []
            ref_np = ref_out.cpu().numpy()
            perr = None
            for rep in range(4):                                # call 0 = first full-size call of the process (cold pools)
                t0 = time.perf_counter()
                res = nrb.reduce_noise(y=ynp, sr=SR, stationary=True, n_fft=1024, hop_length=256)
                calls.append(time.perf_counter() - t0)
                if perr is None:
                    perr = float(np.abs(res - ref_np).max())
                del res                                         # a caller that keeps every result gets fresh buffers instead
            dt = sorted(calls[1:])[len(calls[1:]) // 2]
            line["e2e_numpy"] = {"value": C * n / dt, "unit": UNIT, "ms_per_call": dt * 1e3,
                                 "first_call_ms": calls[0] * 1e3, "calls_ms": [c * 1e3 for c in calls],
                                 "call": "noisereduce_b200.reduce_noise(y=float32[64, 28.8M] pageable ndarray, stationary=True)",
                                 "includes": "noise statistics, staging of the pageable input through pinned slabs, H2D / D2H, result array",
                                 "note": "value = median of calls 2-4: the result array is leased from the library's pinned-buffer pool "
                                         "(b200gate_host_alloc), which the first call has to fill (first_call_ms)",
                                 "parity_vs_device_path": perr}
            del ynp, ref_np
        except Exception as exc:
            line["e2e_numpy"] = {"value": None, "error": repr(exc)[:200]}
        try:
            line["parity"] = same_run_parity(np, torch, dg, x, out)
        except Exception as exc:
            line["parity"] = {"error": repr(exc)[:200]}
        # ---- BASELINE configs 3 and 4 -----------------------------------------------------------------
        extra = {}
        try:
            dg3 = DeviceGate(sr=SR, stationary=False, n_fft=2048, workspace_limit_bytes=72e9)   # all 3072 units in one batch (66 GB of 180)
            for _ in range(2):
                dg3.run(x, out)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                dg3.run(x, out)
            a1.record()
            torch.cuda.synchronize()
            ms3 = a0.elapsed_time(a1) / 3
            s3 = dg3.gate.stats()
            extra["config3"] = {"workload": "64ch x 10min 48kHz non-stationary n_fft=2048 (configs[2])",
                                "value": C * n / (ms3 * 1e-3), "unit": UNIT, "ms_per_step": ms3,
                                "kernel_ms": {"analysis": s3["k1_ms"], "follower+smoothing": s3["smooth_ms"], "synthesis": s3["k2_ms"]},
                                "roofline_whole_step_frac": ALGO_BYTES_PER_SAMPLE * C * n / (ms3 * 1e-3) / 1e9 / peak}
            del dg3
        except Exception as exc:
            extra["config3"] = {"value": None, "error": repr(exc)[:200]}
        try:
            from noisereduce_b200.torchgate import TorchGate
            g4 = torch.Generator(device=device).manual_seed(1234)
            x4 = 0.05 * torch.randn((256, 160000), device=device, generator=g4)
            tg = TorchGate(sr=16000).to(device)
            with torch.no_grad():
                for _ in range(3):
                    tg(x4)
                torch.cuda.synchronize()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(10):
                    tg(x4)
                a1.record()
                torch.cuda.synchronize()
            ms4 = a0.elapsed_time(a1) / 10
            extra["config4"] = {"workload": "TorchGate(sr=16000) forward, batch 256 x 10 s (configs[3])",
                                "value": 256 * 160000 / (ms4 * 1e-3), "unit": UNIT, "ms_per_forward": ms4,
                                "roofline_whole_step_frac": ALGO_BYTES_PER_SAMPLE * 256 * 160000 / (ms4 * 1e-3) / 1e9 / peak}
            del x4, tg
        except Exception as exc:
            extra["config4"] = {"value": None, "error": repr(exc)[:200]}
        if not args.no_cpu_baseline:
            try:
                r3 = cpu_reference_run(1, 0, channels=8, stationary=False, n_fft=2048, with_single_job=False)
                extra["config3"]["cpu_baseline"] = {k: r3[k] for k in ("value", "unit", "cores", "kind", "sample", "n_jobs")}
            except Exception as exc:
                extra["config3"]["cpu_baseline"] = {"value": None, "error": repr(exc)[:160]}
            extra["config4"]["cpu_baseline"] = torchgate_cpu_leg()
        line["configs_extra"] = extra
    if n_gpus == 1 and not args.no_cpu_baseline:
        r = cpu_reference_run(1, 1)
        line["cpu_baseline"] = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample", "n_jobs", "host_cores",
                                                  "busy_workers_max", "versions", "n_jobs_1_value") if k in r}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
