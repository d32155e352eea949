"""Parity on a real B200 (-m gpu), through the C ABI of the nvcc-built libb200gate.so."""
import numpy as np
import pytest

from noisereduce_b200 import _cabi
from oracle import spectral_gate_oracle as O
from tests import parity_cases as P
from tests.golden import fixtures as golden
from tests.synth_host import synth_small

pytestmark = pytest.mark.gpu
SR = 16000


@pytest.fixture(scope="module")
def lib():
    return _cabi.library()          # the product library; raises if it was not built


def _assert_stationary(res):
    assert res["spec_err"] < P.SPEC_TOL, res
    assert res["mask0_mismatch"] == 0, res
    assert res["mask_err"] < P.MASK_TOL, res
    assert res["out_relinf"] < P.OUT_TOL_TIGHT, res
    assert res["stats"]["bins_unresolved"] == 0 and res["stats"]["rowfloor_ambiguous"] == 0, res
    assert res["thresh_err_db"] < P.THRESH_TOL_DB, res


def test_small_cases_match_simulator_suite(lib):
    y = synth_small(C=2, n=12000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=5000, padding=600)
    for unit in [(1, 1), (2, 0), (0, 1)]:
        _assert_stationary(P.check_stationary(lib, y, cfg, tap_unit=unit))
    cfg = O.GateConfig(sr=SR, stationary=True, prop_decrease=0.8)
    _assert_stationary(P.check_stationary(lib, y[:1, :7000], cfg, y_noise=y[:1, 1000:5000]))
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=0)
    _assert_stationary(P.check_stationary(lib, y[:1, :6000], cfg, tap_unit=(2, 0)))
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=None, padding=300)
    res = P.check_stationary(lib, y[:1, :5000], cfg, debug_guard_scale=100000)
    assert res["stats"]["bins_rechecked_fp64"] > 100
    _assert_stationary(res)


def test_config2_shaped_chunks_mask_bit_exact(lib):
    """48 kHz, default chunk_size / padding (config 2 geometry: T = 2579 frames, 11 x 19 filter),
    3 channels x 1.3 M samples = 3 chunks: first / interior / last chunk taps."""
    sr = 48000
    rng = np.random.default_rng(1000)
    n = 1_300_000
    t = np.arange(n) / sr
    y = 0.05 * rng.standard_normal((3, n))
    for c in range(3):
        y[c] += 0.25 * ((t % 2.0) < 0.5) * np.sin(2 * np.pi * 440 * 2 ** (c / 12) * t)
    y = y.astype(np.float32)
    cfg = O.GateConfig(sr=sr, stationary=True)
    worst = 0.0
    for unit in [(0, 0), (1, 2), (2, 1)]:
        res = P.check_stationary(lib, y, cfg, tap_unit=unit)
        _assert_stationary(res)
        assert res["T"] == 2579
        worst = max(worst, res["out_relinf"])
    # the default path runs the dual kernels (two channels per warp); the one-unit-per-warp kernels (path_flags 16)
    # must agree with it and with the oracle
    for flags in (16,):
        alt = P.check_stationary(lib, y, cfg, tap_unit=(1, 2), path_flags=flags)
        _assert_stationary(alt)
        assert P.relinf(res["out"], alt["out"]) < P.OUT_TOL_TIGHT
    print("config-2 geometry: worst rel-inf", worst, "rechecked", res["stats"]["bins_rechecked_fp64"])
    # the library's own thresholds, end to end
    res = P.check_stationary(lib, y, cfg, tap_unit=(1, 0), inject_thresh=False)
    assert res["out_relinf"] < P.OUT_TOL
    assert res["mask0_mismatch"] <= 2          # threshold noise of the reference's float32 noise STFT


def test_nonstationary(lib, golden_dir):
    import noisereduce_b200 as nr
    y = synth_small(C=2, n=12000)
    cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=5000, padding=600, time_constant_s=0.2)
    for unit in [(1, 1), (0, 0), (2, 1)]:
        res = P.check_nonstationary(lib, y, cfg, tap_unit=unit)
        assert res["spec_err"] < P.SPEC_TOL and res["mask_err"] < P.MASK_TOL_NONSTAT, res
        assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5, res
    # config-3-like geometry at n_fft=1024: 48 kHz, default chunking, 2 s time constant
    sr = 48000
    rng = np.random.default_rng(1001)
    n = 1_300_000
    t = np.arange(n) / sr
    yy = (0.05 * rng.standard_normal((2, n)) + 0.25 * ((t % 2.0) < 0.5) * np.sin(2 * np.pi * 440 * t)).astype(np.float32)
    cfg = O.GateConfig(sr=sr, stationary=False)
    res = P.check_nonstationary(lib, yy, cfg, tap_unit=(1, 1))
    assert res["mask_err"] < P.MASK_TOL_NONSTAT and res["out_relinf"] < P.OUT_TOL_TIGHT * 5, res
    # golden: reference outputs
    s = golden.load(golden_dir, "synth_small")
    out = nr.reduce_noise(y=s["y"], sr=int(s["sr"]), stationary=False, chunk_size=12000, padding=1500)
    assert P.relinf(out, s["out_nonstat_chunked"]) < P.OUT_TOL
    f = golden.load(golden_dir, "fish_cfg1")
    out = nr.reduce_noise(y=f["y"], sr=int(f["sr"]), stationary=False)
    assert np.abs(out.astype(np.int32) - f["out_nonstationary"].astype(np.int32)).max() <= 1


def test_nonstationary_n_fft_2048_config3(lib, golden_dir):
    """Config 3 geometry: 48 kHz, n_fft=2048 (hop 512, F=1025, T=1290 per chunk, filter 21 x 9)."""
    import noisereduce_b200 as nr
    sr = 48000
    rng = np.random.default_rng(1002)
    n = 1_300_000
    t = np.arange(n) / sr
    y = (0.05 * rng.standard_normal((2, n)) + 0.25 * ((t % 2.0) < 0.5) * np.sin(2 * np.pi * 523.25 * t)).astype(np.float32)
    cfg = O.GateConfig(sr=sr, stationary=False, n_fft=2048)
    for unit in [(0, 0), (1, 1), (2, 0)]:
        res = P.check_nonstationary(lib, y, cfg, tap_unit=unit)
        assert res["T"] == 1290
        assert res["spec_err"] < P.SPEC_TOL and res["mask_err"] < P.MASK_TOL_NONSTAT, res
        assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5, res
    s = golden.load(golden_dir, "synth_small")
    out = nr.reduce_noise(y=s["y"].astype(np.float64), sr=int(s["sr"]), stationary=False, n_fft=2048,
                          time_constant_s=0.5, prop_decrease=0.9)
    assert out.dtype == np.float64 and P.relinf(out, s["out_nonstat_2048_f64"]) < P.OUT_TOL
    # the forced paths: tap-loop smoothing (128), stored forward sweep (64)
    for flags in (128, 64):
        res = P.check_nonstationary(lib, y, cfg, tap_unit=(1, 0), path_flags=flags)
        assert res["spec_err"] < P.SPEC_TOL and res["mask_err"] < P.MASK_TOL_NONSTAT, (flags, res)
        assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5, (flags, res)


def test_pooled_result_buffers(lib):
    """Large results of the numpy surface come back in page-locked memory leased from the library's pool
    (b200gate_host_alloc): same values as an ordinary array, the lease returns with the last view, and the next call of
    the same size gets the same buffer back."""
    import gc
    import noisereduce_b200 as nr
    sr = 48000
    rng = np.random.default_rng(7)
    y = (0.05 * rng.standard_normal((8, 1_300_000))).astype(np.float32)           # 41.6 MB > PINNED_RESULT_MIN_BYTES
    a = nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=1024, hop_length=256)
    assert _cabi._pinned_leased_bytes >= a.nbytes
    ptr_a = a.ctypes.data
    plain = np.empty_like(y)
    g = _cabi.Gate(lib=lib, **P.gate_params(O.GateConfig(sr=sr, stationary=True, n_fft=1024, hop_length=256)))
    g.noise_stats_host(y)
    g.run_host(y, out=plain)
    g.close()
    assert np.array_equal(a, plain)
    view = a[:, 100:200]
    del a
    gc.collect()
    assert _cabi._pinned_leased_bytes >= y.nbytes and float(np.abs(view).max()) >= 0.0
    del view
    gc.collect()
    assert _cabi._pinned_leased_bytes == 0
    b = nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=1024, hop_length=256)
    assert b.ctypes.data == ptr_a and np.array_equal(b, plain)


def test_golden_fish_and_small(lib, golden_dir):
    import noisereduce_b200 as nr
    f = golden.load(golden_dir, "fish_cfg1")
    out = nr.reduce_noise(y=f["y"], sr=int(f["sr"]), stationary=True)
    assert out.dtype == np.int16 and out.shape == f["y"].shape
    assert np.abs(out.astype(np.int32) - f["out_stationary"].astype(np.int32)).max() <= 1      # <= 1 LSB
    yf = (f["y"] / 32768).astype(np.float32)
    out = nr.reduce_noise(y=yf, sr=int(f["sr"]), stationary=True)
    assert P.relinf(out, f["out_stationary_f32"]) < P.OUT_TOL
    s = golden.load(golden_dir, "synth_small")
    kw = dict(chunk_size=12000, padding=1500)
    y, sr = s["y"], int(s["sr"])
    assert P.relinf(nr.reduce_noise(y=y, sr=sr, stationary=True, **kw), s["out_stat_chunked"]) < P.OUT_TOL
    assert P.relinf(nr.reduce_noise(y=y, sr=sr, stationary=True, y_noise=y[:, 3000:11000], prop_decrease=0.8, **kw),
                    s["out_stat_ynoise_p08"]) < P.OUT_TOL
    assert P.relinf(nr.reduce_noise(y=y[0], sr=sr, stationary=True), s["out_stat_single_chunk"]) < P.OUT_TOL
    assert P.relinf(nr.reduce_noise(y=y, sr=sr, stationary=True, freq_mask_smooth_hz=None,
                                    time_mask_smooth_ms=None, **kw), s["out_stat_nosmooth"]) < P.OUT_TOL


def test_get_traces_subranges_golden(lib, golden_dir):
    """SpectralGate.get_traces(start_frame, end_frame) against reference outputs (base.py:167-226): only
    the selected units run, and the result equals the reference's chunk-grid / single-chunk branches."""
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    g = golden.load(golden_dir, "synth_traces")
    y = synth_small()
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, clip_noise_stationary=True, n_fft=1024, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500, time_mask_smooth_ms=50,
                tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1)
    sg = SpectralGateStationary(y=y, sr=16000, chunk_size=12000, padding=1500, **args)
    for key, (a, b, units) in {"chunks_13000_28000": (13000, 28000, 4), "chunks_500_24500": (500, 24500, 6),
                               "single_to_9000": (4000, 9000, 2)}.items():
        out = sg.get_traces(a, b)
        assert out.shape == g[key].shape and P.relinf(out, g[key]) < P.OUT_TOL, key
        assert sg._gate.stats()["units"] == units, key
    sg = SpectralGateStationary(y=y, sr=16000, chunk_size=None, padding=1500, **args)
    out = sg.get_traces(None, 29000)
    assert P.relinf(out, g["single_to_29000_nochunk"]) < P.OUT_TOL
    # device-resident rows through the same range selection
    import torch
    gate = SpectralGateStationary(y=y, sr=16000, chunk_size=12000, padding=1500, **args)._gate
    x = torch.from_numpy(y).cuda()
    o = torch.full_like(x, 7.0)
    gate.set_range(1, 1, 1)
    gate.run_device(x.data_ptr(), o.data_ptr(), np.float32, 2, 30000, 30000, 30000)
    torch.cuda.synchronize()
    gate.set_range(0)
    o = o.cpu().numpy()
    assert np.all(o[:, :12000] == 7.0) and np.all(o[:, 24000:] == 7.0)          # untouched outside chunk 1
    ref = O.reduce_noise(y, 16000, cfg=O.GateConfig(sr=16000, stationary=True, chunk_size=12000, padding=1500))
    assert P.relinf(o[:, 12000:24000], ref[:, 12000:24000]) < P.OUT_TOL


def test_device_pointer_path_and_properties(lib):
    """Device-resident tensors through the same C call; linearity-in-scale and chunk independence."""
    import torch
    from noisereduce_b200.device import DeviceGate
    sr = 48000
    g = torch.Generator(device="cuda").manual_seed(7)
    x = 0.05 * torch.randn((4, 2_000_000), device="cuda", generator=g)
    dg = DeviceGate(sr=sr, stationary=True)
    dg.noise_stats(x)
    y = dg.run(x)
    torch.cuda.synchronize()
    ref = O.reduce_noise(x[:1].cpu().numpy(), sr, cfg=O.GateConfig(sr=sr, stationary=True),
                         thresh_override=dg.gate.noise_threshold(), return_float64=True)
    assert P.relinf(y[:1].cpu().numpy(), ref) < P.OUT_TOL_TIGHT
    # idempotent launch: same input -> bit-identical output (no races in the overlap-add seams)
    y2 = dg.run(x)
    assert torch.equal(y, y2)
    # native int16 / float64 device rows: the kernels load and store the caller's dtype
    xi = (x[:2, :1_300_000] * 20000).to(torch.int16)
    dgi = DeviceGate(sr=sr, stationary=True)
    dgi.noise_stats(xi)
    yi = dgi.run(xi)
    assert yi.dtype == torch.int16
    refi = O.reduce_noise(xi.cpu().numpy(), sr, cfg=O.GateConfig(sr=sr, stationary=True),
                          thresh_override=dgi.gate.noise_threshold())
    assert np.abs(yi.cpu().numpy().astype(np.int32) - refi.astype(np.int32)).max() <= 1
    xd = x[:1, :700_000].double()
    dgd = DeviceGate(sr=sr, stationary=False)
    yd = dgd.run(xd)
    refd = O.reduce_noise(xd.cpu().numpy(), sr, cfg=O.GateConfig(sr=sr, stationary=False), return_float64=True)
    assert yd.dtype == torch.float64 and P.relinf(yd.cpu().numpy(), refd) < P.OUT_TOL_TIGHT * 5


def test_torchgate_surface(lib, golden_dir):
    """Config 4 surface: CUDA tensors through TorchGate.forward, vs the reference's own outputs
    (tests/golden/torchgate_small.npz) and the float64 oracle."""
    import torch
    from noisereduce_b200.torchgate import TorchGate
    from oracle import torchgate_oracle as TO
    g = golden.load(golden_dir, "torchgate_small")
    x = torch.from_numpy(g["x"]).cuda()
    sr = int(g["sr"])
    tol = 2e-5          # FP32 path vs the reference's float32 / float64 runs (its own f32-vs-f64 gap is 2.5e-7)
    y = TorchGate(sr=sr).to("cuda")(x)
    assert y.is_cuda and y.dtype == torch.float32 and tuple(y.shape) == tuple(g["out_stat_f32"].shape)
    assert P.relinf(y.cpu().numpy(), g["out_stat_f64"]) < tol
    assert P.relinf(y.cpu().numpy(), g["out_stat_f32"]) < tol
    y = TorchGate(sr=sr, nonstationary=True)(x)
    assert P.relinf(y.cpu().numpy(), g["out_nonstat_f64"]) < tol
    y = TorchGate(sr=sr, prop_decrease=0.7)(x.double(), x[:1, :6000].double())
    assert y.dtype == torch.float64
    assert P.relinf(y.cpu().numpy(), g["out_stat_xn_p07_f64"]) < tol
    # config-4 shaped batch (subset of rows checked against the oracle)
    gen = torch.Generator(device="cuda").manual_seed(1234)
    xb = 0.05 * torch.randn((32, 160000), device="cuda", generator=gen)
    t = torch.arange(160000, device="cuda") / 16000
    xb += 0.2 * torch.sin(2 * torch.pi * 700 * t) * ((t % 1.0) < 0.3)
    tg = TorchGate(sr=16000)
    yb = tg(xb)
    torch.cuda.synchronize()
    assert tuple(yb.shape) == (32, 160000)
    for r in (0, 31):
        ref = TO.torchgate_forward(xb[r:r + 1].cpu().numpy().astype(np.float64), 16000,
                                   window=torch.hann_window(1024).numpy())
        assert P.relinf(yb[r:r + 1].cpu().numpy(), ref) < 1e-4


def test_batching_slabs_and_config5_geometry(lib):
    """Workspace batching / host slab streaming at realistic sizes, and config-5 chunking (60 s chunks,
    T = 11485): results must not depend on how units are batched, and must match the oracle."""
    import noisereduce_b200 as nr
    sr = 48000
    rng = np.random.default_rng(1003)
    n = 6_500_000                                      # > 2 chunks of 2.88 M samples
    t = np.arange(n) / sr
    y = (0.05 * rng.standard_normal((2, n)) + 0.25 * ((t % 2.0) < 0.5) * np.sin(2 * np.pi * 660 * t)).astype(np.float32)
    kw = dict(chunk_size=2_880_000, padding=30000)
    cfg = O.GateConfig(sr=sr, stationary=True, **kw)
    res = P.check_stationary(lib, y, cfg, tap_unit=(1, 1))
    assert res["T"] == 11485
    _assert_stationary(res)
    # default chunking, tiny workspace -> many batches / slabs; identical to the one-batch result
    cfg = O.GateConfig(sr=sr, stationary=True)
    a = P.check_stationary(lib, y[:, :3_000_000], cfg, tap_unit=(2, 1))
    b = P.check_stationary(lib, y[:, :3_000_000], cfg, tap_unit=(2, 1), workspace_limit_bytes=30.0e6)
    _assert_stationary(a)
    assert b["stats"]["kernel_launches"] > a["stats"]["kernel_launches"]
    assert np.array_equal(a["out"], b["out"])
    # int16 host input streams through the raw-dtype slab pipeline
    yi = (y[:, :2_000_000] * 20000).astype(np.int16)
    out = nr.reduce_noise(y=yi, sr=sr, stationary=True)
    ref = O.reduce_noise(yi, sr, cfg=O.GateConfig(sr=sr, stationary=True))
    assert out.dtype == np.int16 and np.abs(out.astype(np.int32) - ref.astype(np.int32)).max() <= 1


def test_reference_test_suite_scenarios(lib, golden_dir):
    """test_reduction.py:6-56 of the reference, through reduce_noise() on the GPU, against the oracle."""
    import noisereduce_b200 as nr
    f = golden.load(golden_dir, "fish_cfg1")
    sr = int(f["sr"])
    for name, y, kw in P.reference_test_suite_scenarios(f["y"], sr):
        out = nr.reduce_noise(y=y, sr=sr, **kw)
        cfg_kw = {k: v for k, v in kw.items() if k != "y_noise"}
        ref = O.reduce_noise(y, sr, y_noise=kw.get("y_noise"), cfg=O.GateConfig(sr=sr, **cfg_kw))
        assert out.dtype == np.float64 and out.shape == y.shape, name
        assert P.relinf(out, ref) < (P.OUT_TOL_TIGHT if kw["stationary"] else 10 * P.OUT_TOL_TIGHT), name


def test_general_geometry_family_golden_and_stages(lib, golden_dir):
    """STFT geometries off the default run on the float64 general family (gate_generic.cuh): reference
    outputs (tests/golden/synth_geometry.npz), stage taps against the oracle, and the tuned n_fft=1024
    kernels cross-checked against the general family on the same input."""
    import noisereduce_b200 as nr
    from tests.test_oracle_golden import GEOMETRY_CASES, NON_POW2_KEYS, geometry_input
    g = golden.load(golden_dir, "synth_geometry")
    for key, (kw, dt) in GEOMETRY_CASES.items():
        if key in NON_POW2_KEYS:
            continue                                   # test_non_power_of_two_n_fft_golden
        y = geometry_input(dt)
        out = nr.reduce_noise(y=y, sr=16000, chunk_size=12000, padding=1500, **kw)
        assert out.dtype == g[key].dtype and out.shape == g[key].shape, key
        if dt == np.int16:
            assert np.abs(out.astype(np.int64) - g[key].astype(np.int64)).max() <= 1, key
        else:
            assert P.relinf(out, g[key]) < P.OUT_TOL_TIGHT, key
    y = synth_small(C=3, n=40000)
    for geo in (dict(n_fft=512, win_length=400, hop_length=100), dict(n_fft=4096, win_length=2048, hop_length=512),
                dict(n_fft=64, win_length=63, hop_length=20)):
        cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=15000, padding=2000, freq_mask_smooth_hz=None,
                           time_mask_smooth_ms=None if geo["n_fft"] == 4096 else 50, **geo)
        if geo["n_fft"] == 64:
            cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=15000, padding=2000, freq_mask_smooth_hz=1000,
                               time_mask_smooth_ms=20, **geo)
        r = P.check_stationary(lib, y, cfg, tap_unit=(1, 2))
        assert r["mask0_mismatch"] == 0 and r["spec_err"] < 2e-7 and r["mask_err"] < 2e-7 and r["out_relinf"] < 2e-7, (geo, r)
        cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=15000, padding=2000, time_constant_s=0.3,
                           freq_mask_smooth_hz=cfg.freq_mask_smooth_hz, time_mask_smooth_ms=cfg.time_mask_smooth_ms, **geo)
        r = P.check_nonstationary(lib, y, cfg, tap_unit=(2, 0))
        assert r["spec_err"] < 2e-7 and r["mask_err"] < 2e-7 and r["out_relinf"] < 2e-7, (geo, r)
    # the tuned FP32 kernels against the float64 family, same library, same thresholds
    y = synth_small(C=4, n=200000)
    a = nr.reduce_noise(y=y, sr=SR, stationary=True, chunk_size=60000, padding=3000)
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, clip_noise_stationary=True, n_fft=1024, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500, time_mask_smooth_ms=50,
                tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1, chunk_size=60000, padding=3000)
    sg = SpectralGateStationary(y=y, sr=SR, **args)
    import noisereduce_b200._cabi as cabi
    gen = cabi.Gate(lib, **{**sg._gate_params(), "stationary": 1, "n_std_thresh": 1.5, "clip_noise": 1, "path_flags": 4})
    gen.set_noise_threshold(sg.noise_thresh)
    b = gen.run_host(np.ascontiguousarray(y))
    assert P.relinf(a, b) < P.OUT_TOL_TIGHT


def test_torchgate_general_geometry_golden(lib, golden_dir):
    """TorchGate off the default STFT geometry on the GPU (general family, torch framing) against reference outputs."""
    import torch
    from noisereduce_b200.torchgate import TorchGate
    from tests.synth_host import synth_torchgate
    from tests.test_oracle_golden import NON_POW2_KEYS, TG_GEOMETRY_CASES
    g = golden.load(golden_dir, "torchgate_geometry")
    x = synth_torchgate()[:2, :12000]
    for key, (kw, xn_idx, dt) in TG_GEOMETRY_CASES.items():
        if key in NON_POW2_KEYS:
            continue
        xt = torch.from_numpy(x.astype(dt)).cuda()
        xn = None if xn_idx is None else xt[xn_idx]
        y = TorchGate(sr=16000, **kw)(xt, xn)
        assert y.dtype == xt.dtype and tuple(y.shape) == g[key].shape, key
        assert P.relinf(y.cpu().numpy(), g[key]) < 5e-5, key


def test_non_power_of_two_n_fft_golden(lib, golden_dir):
    """n_fft = 400 / 441 / 1000: Bluestein's chirp-z inside the general family (two length-M radix-2 transforms in
    shared memory), both surfaces, against reference outputs; stage taps against the oracle."""
    import torch
    import noisereduce_b200 as nr
    from noisereduce_b200.torchgate import TorchGate
    from tests.synth_host import synth_torchgate
    from tests.test_oracle_golden import GEOMETRY_CASES, NON_POW2_KEYS, TG_GEOMETRY_CASES, geometry_input
    g = golden.load(golden_dir, "synth_geometry")
    for key, (kw, dt) in GEOMETRY_CASES.items():
        if key in NON_POW2_KEYS:
            out = nr.reduce_noise(y=geometry_input(dt), sr=16000, chunk_size=12000, padding=1500, **kw)
            assert out.shape == g[key].shape and P.relinf(out, g[key]) < P.OUT_TOL_TIGHT, key
    y = synth_small(C=2, n=30000)
    for geo in (dict(n_fft=400), dict(n_fft=441, win_length=441, hop_length=110), dict(n_fft=3000, win_length=2000, hop_length=500)):
        ms = 50 if geo["n_fft"] < 3000 else None
        cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=12000, padding=1500, time_mask_smooth_ms=ms, **geo)
        r = P.check_stationary(lib, y, cfg, tap_unit=(1, 1))
        assert r["mask0_mismatch"] == 0 and r["spec_err"] < 2e-7 and r["mask_err"] < 2e-7 and r["out_relinf"] < 2e-7, (geo, r)
        cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=12000, padding=1500, time_constant_s=0.3, time_mask_smooth_ms=ms, **geo)
        r = P.check_nonstationary(lib, y, cfg, tap_unit=(2, 0))
        assert r["spec_err"] < 2e-7 and r["mask_err"] < 2e-7 and r["out_relinf"] < 2e-7, (geo, r)
    gt = golden.load(golden_dir, "torchgate_geometry")
    x = synth_torchgate()[:2, :12000]
    for key, (kw, xn_idx, dt) in TG_GEOMETRY_CASES.items():
        if key in NON_POW2_KEYS:
            xt = torch.from_numpy(x.astype(dt)).cuda()
            yt = TorchGate(sr=16000, **kw)(xt)
            assert tuple(yt.shape) == gt[key].shape and P.relinf(yt.cpu().numpy(), gt[key]) < 5e-5, key


def test_edge_cases_like_the_reference(lib, golden_dir):
    """The edge cases pinned by tests/golden/edge_cases.npz (outputs of the unmodified reference) on the GPU."""
    import noisereduce_b200 as nr
    from tests.test_cusim_parity import _replay_edge_cases
    _replay_edge_cases(nr, golden_dir)
