"""Kernel-logic parity on the CPU simulator build (tests/cusim) -- runs in the GPU-less container.

These run the PRODUCT's .cu sources (compiled by g++ against the cusim shim) on tiny inputs and
compare them with oracle/.  They guard indexing / barrier / shuffle logic and the host planner; the
real-hardware parity tests are tests/test_gpu_parity.py (-m gpu).
"""
import numpy as np
import pytest

from noisereduce_b200 import _cabi
from oracle import spectral_gate_oracle as O
from tests import parity_cases as P
from tests.cusim_util import cusim_library
from tests.golden import fixtures as golden
from tests.synth_host import synth_small

SR = 16000


@pytest.fixture(scope="module")
def lib():
    return cusim_library()


def _assert_stationary(res, exact_bits=True):
    assert res["spec_err"] < P.SPEC_TOL
    if exact_bits:
        assert res["mask0_mismatch"] == 0
    assert res["mask_err"] < P.MASK_TOL
    assert res["out_relinf"] < P.OUT_TOL_TIGHT
    assert res["stats"]["bins_unresolved"] == 0
    assert res["stats"]["rowfloor_ambiguous"] == 0
    assert res["thresh_err_db"] < P.THRESH_TOL_DB


def test_stationary_chunked_two_channels(lib):
    y = synth_small(C=2, n=12000)
    for pad in (600, 601):                              # 601: every sample row starts off a 16-byte boundary
        cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=5000, padding=pad)
        res = P.check_stationary(lib, y, cfg, tap_unit=(1, 1))
        _assert_stationary(res)
        assert res["stats"]["units"] == 6 and res["mask0_on_frac"] > 0.05
        # last chunk (shorter valid span) and first chunk (left zero padding)
        _assert_stationary(P.check_stationary(lib, y, cfg, tap_unit=(2, 0)))
        _assert_stationary(P.check_stationary(lib, y, cfg, tap_unit=(0, 1)))


def test_spectrum_cache_paths(lib):
    """k1 / k1n store the packed spectra and k2 loads them (no second forward FFT), checked against the oracle."""
    y = synth_small(C=2, n=12000)
    for stationary in (True, False):
        cfg = O.GateConfig(sr=SR, stationary=stationary, chunk_size=5000, padding=600, time_constant_s=0.2, prop_decrease=0.9)
        chk = P.check_stationary if stationary else P.check_nonstationary
        a = chk(lib, y, cfg, tap_unit=(1, 1))
        assert a["mask_err"] < P.MASK_TOL_NONSTAT and a["out_relinf"] < P.OUT_TOL_TIGHT * 5
        if stationary:
            assert a["mask0_mismatch"] == 0
    # odd first frame of a run, single chunk, tiny padding: pair alignment of the cached spectra
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=0)
    _assert_stationary(P.check_stationary(lib, y[:1, :7000], cfg, tap_unit=(2, 0)))


def test_pipelined_host_path_one_chunk_per_slab(lib):
    """Host float32 input is streamed slab by slab (H2D / kernels / D2H on three streams); a tiny
    workspace limit forces one chunk per slab so slab seams and buffer recycling are exercised."""
    y = synth_small(C=2, n=23000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=4000, padding=600)
    res = P.check_stationary(lib, y, cfg, tap_unit=(3, 1), workspace_limit_bytes=300000.0)
    _assert_stationary(res)
    assert res["stats"]["units"] == 12 and res["stats"]["kernel_launches"] >= 6 * 4
    cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=4000, padding=600, time_constant_s=0.3)
    res = P.check_nonstationary(lib, y, cfg, tap_unit=(5, 0), workspace_limit_bytes=500000.0)
    assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5


def test_stationary_own_thresholds_end_to_end(lib):
    y = synth_small(C=2, n=9000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=4000, padding=500)
    res = P.check_stationary(lib, y, cfg, tap_unit=(0, 0), inject_thresh=False)
    assert res["thresh_err_db"] < P.THRESH_TOL_DB
    assert res["out_relinf"] < P.OUT_TOL


def test_stationary_single_chunk_blend_and_ynoise(lib):
    y = synth_small(C=1, n=7000)
    cfg = O.GateConfig(sr=SR, stationary=True, prop_decrease=0.8)          # defaults: one padded chunk
    res = P.check_stationary(lib, y, cfg, y_noise=y[:, 1000:5000])
    _assert_stationary(res)
    assert res["stats"]["units"] == 1


def test_stationary_no_smoothing_and_tiny_padding(lib):
    y = synth_small(C=1, n=6000)
    cfg = O.GateConfig(sr=SR, stationary=True, freq_mask_smooth_hz=None, time_mask_smooth_ms=None,
                       chunk_size=2500, padding=100)      # padding < hop: tail zeros + edge overlap-add norms
    res = P.check_stationary(lib, y, cfg, tap_unit=(1, 0))
    _assert_stationary(res)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=0)
    _assert_stationary(P.check_stationary(lib, y, cfg, tap_unit=(2, 0)))


def test_smoothing_kernel_variants(lib):
    """packed dp4a kernel with 3 / 6 / 9 tap words, and the generic fallback for long time extents."""
    y = synth_small(C=1, n=7000)
    for hz, ms in [(100, 50), (300, 100), (500, 200), (200, 250)]:    # nf = 3, 9, 16, 6; nt = 3, 6, 12, 15
        cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=3000, padding=500, freq_mask_smooth_hz=hz,
                           time_mask_smooth_ms=ms, prop_decrease=0.9)
        res = P.check_stationary(lib, y, cfg, tap_unit=(1, 0))
        _assert_stationary(res)


def test_fp64_redecision_path_gives_same_bits(lib):
    y = synth_small(C=1, n=5000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=None, padding=300)
    res = P.check_stationary(lib, y, cfg, debug_guard_scale=100000)
    assert res["stats"]["bins_rechecked_fp64"] > 100        # the knob forced many bins through FP64
    _assert_stationary(res)


def test_top_db_row_floor(lib):
    # a steady loud tone sits > 80 dB above the noise threshold of its bin: the whole row is lifted
    n = 6000
    t = np.arange(n) / SR
    rng = np.random.default_rng(5)
    y = (1e-5 * rng.standard_normal(n) + 0.9 * np.sin(2 * np.pi * 1000 * t)).astype(np.float32)[None, :]
    noise = (1e-5 * rng.standard_normal(4000)).astype(np.float32)[None, :]
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=None, padding=300)
    res = P.check_stationary(lib, y, cfg, y_noise=noise)
    assert res["stats"]["rowfloor_flags"] > 0
    _assert_stationary(res)


def test_int16_and_float64_io(lib):
    y = synth_small(C=2, n=6000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=400)
    yi = (y * 20000).astype(np.int16)
    res = P.check_stationary(lib, yi, cfg)
    assert res["out_dtype_ok"] and res["out_max_lsb"] <= 1
    res = P.check_stationary(lib, y.astype(np.float64), cfg)
    assert res["out_dtype_ok"] and res["out_relinf"] < P.OUT_TOL_TIGHT


def test_nonstationary_chunked(lib):
    y = synth_small(C=2, n=12000)
    cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=5000, padding=600, time_constant_s=0.2)
    for unit in [(1, 1), (0, 0), (2, 1)]:
        res = P.check_nonstationary(lib, y, cfg, tap_unit=unit)
        assert res["spec_err"] < P.SPEC_TOL and res["mask_err"] < P.MASK_TOL_NONSTAT
        assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5
    # defaults (2 s time constant, one padded chunk), prop_decrease < 1, no smoothing
    cfg = O.GateConfig(sr=SR, stationary=False, prop_decrease=0.7)
    res = P.check_nonstationary(lib, y[:1, :7000], cfg)
    assert res["mask_err"] < P.MASK_TOL_NONSTAT and res["out_relinf"] < P.OUT_TOL_TIGHT * 5
    cfg = O.GateConfig(sr=SR, stationary=False, freq_mask_smooth_hz=None, time_mask_smooth_ms=None,
                       chunk_size=3000, padding=200, thresh_n_mult_nonstationary=1.5, sigmoid_slope_nonstationary=5)
    res = P.check_nonstationary(lib, y[:1, :7000], cfg, tap_unit=(1, 0))
    assert res["mask_err"] < P.MASK_TOL_NONSTAT and res["out_relinf"] < P.OUT_TOL_TIGHT * 5


def test_nonstationary_n_fft_2048(lib):
    """config-3 family: one real 2048-sample frame per complex-1024 warp FFT (half-length trick)."""
    y = synth_small(C=2, n=20000)
    cases = [(dict(chunk_size=8000, padding=1200, time_constant_s=0.3), [(1, 1), (0, 0), (2, 0)]),
             (dict(prop_decrease=0.8), [(0, 1)]),
             (dict(chunk_size=7000, padding=100), [(2, 0)])]
    for kw, units in cases:
        cfg = O.GateConfig(sr=SR, stationary=False, n_fft=2048, **kw)
        for unit in units:
            res = P.check_nonstationary(lib, y, cfg, tap_unit=unit)
            assert res["spec_err"] < P.SPEC_TOL and res["mask_err"] < P.MASK_TOL_NONSTAT
            assert res["out_relinf"] < P.OUT_TOL_TIGHT * 5


def test_float_mask_box_smoothing_and_2k_spectrum_cache(lib):
    """k_smooth_box (1 <= nf <= 12: two sliding box sums per row) against the oracle and against the tap-loop
    streaming kernel (path_flags 128); k2c_synthesize_2k (spectra cached by k1n_magnitude_2k) against the oracle.
    The last case has config 3's filter extents (nf 10, nt 4)."""
    y = synth_small(C=2, n=20000)
    cases = [(1024, 40, 20), (1024, 70, 70), (1024, 170, 150), (1024, 330, 40), (1024, 390, 100),
             (2048, 16, 40), (2048, 100, 300), (2048, 160, 130)]
    for n_fft, hz, ms in cases:
        cfg = O.GateConfig(sr=SR, stationary=False, n_fft=n_fft, chunk_size=8000, padding=1200, time_constant_s=0.3,
                           freq_mask_smooth_hz=hz, time_mask_smooth_ms=ms, prop_decrease=0.9)
        a = P.check_nonstationary(lib, y, cfg, tap_unit=(1, 1))
        b = P.check_nonstationary(lib, y, cfg, tap_unit=(1, 1), path_flags=128)
        for r in (a, b):
            assert r["mask_err"] < P.MASK_TOL_NONSTAT and r["out_relinf"] < P.OUT_TOL_TIGHT * 5, (n_fft, hz, ms, r)
    cfg = O.GateConfig(sr=SR, stationary=False, n_fft=2048, chunk_size=7000, padding=600, freq_mask_smooth_hz=160,
                       time_mask_smooth_ms=130)
    for unit in [(0, 0), (2, 1)]:
        r = P.check_nonstationary(lib, y, cfg, tap_unit=unit)
        assert r["spec_err"] < P.SPEC_TOL and r["mask_err"] < P.MASK_TOL_NONSTAT and r["out_relinf"] < P.OUT_TOL_TIGHT * 5
    # the follower with its forward sweep stored (path_flags 64) instead of regenerated, odd batch remainders (T = 17, 30)
    for n, cs in [(4000, 0), (7400, 0)]:
        cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=cs or None, padding=300, time_constant_s=0.5)
        for fl in (0, 64):
            r = P.check_nonstationary(lib, y[:1, :n], cfg, path_flags=fl)
            assert r["mask_err"] < P.MASK_TOL_NONSTAT and r["out_relinf"] < P.OUT_TOL_TIGHT * 5, (n, fl, r)


def test_pooled_result_arrays_lease_lifetime(lib, monkeypatch):
    """_cabi.result_empty: large results are leased from b200gate_host_alloc (plain malloc in the simulator build), stay alive
    through views, return with the last one, respect the budget and fall back to np.empty for small arrays."""
    import gc
    base = _cabi._pinned_leased_bytes
    a = _cabi.result_empty(lib, (4, 10_000_000), np.float32)             # 160 MB
    assert isinstance(a, np.ndarray) and a.shape == (4, 10_000_000) and a.flags.writeable
    assert _cabi._pinned_leased_bytes == base + a.nbytes
    a[:] = 2.0
    v = a[1:3, 5:50]
    del a
    gc.collect()
    assert _cabi._pinned_leased_bytes == base + 160_000_000 and float(v.sum()) == 2.0 * 2 * 45
    del v
    gc.collect()
    assert _cabi._pinned_leased_bytes == base
    small = _cabi.result_empty(lib, (4, 100), np.int16)
    assert small.dtype == np.int16 and _cabi._pinned_leased_bytes == base
    monkeypatch.setenv("B200GATE_PINNED_RESULT_LIMIT", "1000000")         # budget smaller than the request: ordinary memory
    big = _cabi.result_empty(lib, (4, 10_000_000), np.float32)
    assert _cabi._pinned_leased_bytes == base and big.shape == (4, 10_000_000)
    # run_host without `out` takes the same route and returns the gate's result
    y = synth_small(C=2, n=9000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=4000, padding=500)
    g = _cabi.Gate(lib=lib, **P.gate_params(cfg))
    g.noise_stats_host(y)
    out = g.run_host(y)
    ref = np.empty_like(y)
    g.run_host(y, out=ref)
    g.close()
    assert np.array_equal(out, ref)


def _replay_edge_cases(nr, golden_dir):
    """reduce_noise() on the edge cases of tests/golden/edge_cases.py against the reference's stored outputs."""
    import os
    from tests.golden import edge_cases as E
    g = np.load(os.path.join(golden_dir, "edge_cases.npz"))
    for name, (y, kw) in E.cases().items():
        out, ref = nr.reduce_noise(y=y, sr=E.SR, **kw), g[name]
        assert out.shape == ref.shape and out.dtype == ref.dtype, name
        if np.issubdtype(ref.dtype, np.integer):
            assert np.abs(out.astype(np.int64) - ref.astype(np.int64)).max() <= 1, name
        else:
            assert np.array_equal(np.isnan(out), np.isnan(ref)), name           # (all-zero input: the reference returns NaN)
            tol = 1e-3 if ref.dtype == np.float16 else P.OUT_TOL
            assert P.relinf(np.nan_to_num(out), np.nan_to_num(ref)) < tol, name
    for name, (y, kw, exc, msg) in E.refused().items():
        with pytest.raises(exc, match=msg):
            nr.reduce_noise(y=y, sr=E.SR, **kw)


def test_edge_cases_like_the_reference_on_simulator(lib, monkeypatch, golden_dir):
    """Short clips (scipy shrinks the STFT window to a noise clip shorter than it, or refuses), ragged chunks, zero padding,
    non-contiguous views, float16 / int32 / uint8 samples, all-zero and constant input, and the inputs the reference
    refuses -- outputs of the unmodified reference (tests/golden/make_golden_edge.py)."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    import noisereduce_b200 as nr
    _replay_edge_cases(nr, golden_dir)


def test_python_surface_on_simulator(lib, monkeypatch):
    """reduce_noise() host logic (shapes, dtypes, defaults, errors) with the simulator library."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    import noisereduce_b200 as nr
    y = synth_small(C=2, n=6000)
    out = nr.reduce_noise(y=y, sr=SR, stationary=True, chunk_size=2500, padding=400, n_jobs=4, use_tqdm=True)
    ref = O.reduce_noise(y, SR, cfg=O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=400))
    assert out.shape == y.shape and out.dtype == y.dtype
    assert P.relinf(out, ref) < P.OUT_TOL
    flat = nr.reduce_noise(y=y[0], sr=SR, stationary=True)
    assert flat.shape == (6000,)
    out = nr.reduce_noise(y=y, sr=SR, chunk_size=2500, padding=400)          # default: non-stationary
    ref = O.reduce_noise(y, SR, cfg=O.GateConfig(sr=SR, stationary=False, chunk_size=2500, padding=400))
    assert P.relinf(out, ref) < P.OUT_TOL
    with pytest.raises(ValueError, match="Waveform must be in shape"):
        nr.reduce_noise(y=np.zeros((2, 2, 100), np.float32), sr=SR, stationary=True)
    with pytest.raises(ValueError, match="freq_mask_smooth_hz needs to be at least"):
        nr.reduce_noise(y=y, sr=SR, stationary=True, freq_mask_smooth_hz=10)
    with pytest.raises(ValueError, match="n_jobs must be 1"):
        nr.reduce_noise(y=y, sr=SR, stationary=True, use_torch=True, n_jobs=2)
    with pytest.raises(_cabi.GateError, match="unsupported STFT geometry"):
        nr.reduce_noise(y=y, sr=SR, stationary=True, n_fft=5000, time_mask_smooth_ms=200)   # beyond the Bluestein size limit
    with pytest.raises(_cabi.GateError, match="unsupported STFT geometry"):
        nr.reduce_noise(y=y, sr=SR, stationary=True, n_fft=512, win_length=600)


def test_do_filter_plugin_point_on_simulator(lib, monkeypatch):
    """The reference's per-chunk operator interface (base.py:130-160): _read_chunk / filter_chunk /
    _get_filtered_chunk / _do_filter(chunk) on the mirror classes, against the oracle's per-unit gate."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    from noisereduce_b200.spectralgate.nonstationary import SpectralGateNonStationary
    y = synth_small(C=2, n=9000)
    kw = dict(chunk_size=3000, padding=400)
    common = dict(n_fft=1024, win_length=None, hop_length=None, time_constant_s=0.3, freq_mask_smooth_hz=500,
                  time_mask_smooth_ms=50, tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1, **kw)
    sg = SpectralGateStationary(y=y, sr=SR, y_noise=None, n_std_thresh_stationary=1.5, clip_noise_stationary=True, **common)
    cfg = O.GateConfig(sr=SR, stationary=True, **kw)
    info = {}
    full = O.reduce_noise(y, SR, cfg=cfg, info=info, return_float64=True)
    chunk = sg._read_chunk(3000 - 400, 6000 + 400)
    assert chunk.dtype == np.float64 and chunk.shape == (2, 3800)
    assert np.array_equal(chunk, O.read_chunk(y, 2600, 6400))
    filt = sg._do_filter(chunk)
    assert filt.shape == chunk.shape and filt.dtype == chunk.dtype
    for c in range(2):
        ref = O.gate_stationary_unit(chunk[c], sg.noise_thresh, cfg, info["filt"])
        assert P.relinf(filt[c], ref) < P.OUT_TOL
    assert P.relinf(sg._get_filtered_chunk(1), full[:, 3000:6000]) < P.OUT_TOL
    assert P.relinf(sg.filter_chunk(6000, 9000), full[:, 6000:9000]) < P.OUT_TOL
    # the last columns past (Lp // hop) * hop stay zero, as stationary.py:126 leaves them
    assert np.all(filt[:, (3800 // 256) * 256:] == 0)
    ns = SpectralGateNonStationary(y=y, sr=SR, thresh_n_mult_nonstationary=2, sigmoid_slope_nonstationary=10, **common)
    cfg_ns = O.GateConfig(sr=SR, stationary=False, time_constant_s=0.3, **kw)
    info = {}
    full = O.reduce_noise(y, SR, cfg=cfg_ns, info=info, return_float64=True)
    filt = ns._do_filter(chunk)
    for c in range(2):
        assert P.relinf(filt[c], O.gate_nonstationary_unit(chunk[c], cfg_ns, info["filt"])) < P.OUT_TOL
    assert P.relinf(ns._get_filtered_chunk(0), full[:, 0:3000]) < P.OUT_TOL


def test_run_sharded_peer_stores_on_simulator(lib):
    """b200gate_run_sharded (kernel-issued gather): two 'ranks' in one process share host buffers as their peer
    mappings; each writes its channel groups into its own copy and pushes them into the other's; both copies must end
    up equal to the single-gate result, flags carry the epoch."""
    import torch
    from noisereduce_b200.device import DeviceGate
    y = torch.from_numpy(synth_small(C=4, n=7000))
    kw = dict(chunk_size=3000, padding=400)
    ref_gate = DeviceGate(sr=SR, stationary=True, lib=lib, **kw)
    ref_gate.noise_stats(y)
    thr = ref_gate.gate.noise_threshold()
    want = ref_gate.run(y).numpy()
    world, Cl, N = 2, 2, y.shape[1]
    gathered = [np.full((world * Cl, N), np.nan, np.float32) for _ in range(world)]
    flags = [np.zeros(64, np.uint32) for _ in range(world)]
    for rank in range(world):
        dg = DeviceGate(sr=SR, stationary=True, lib=lib, **kw)
        dg.gate.set_noise_threshold(thr)
        x_local = y[rank * Cl: (rank + 1) * Cl].contiguous()
        dg.gate.run_sharded(x_local.data_ptr(), np.float32, Cl, N, N, gathered[rank].ctypes.data,
                            [g.ctypes.data for g in gathered], flags[rank].ctypes.data, [f.ctypes.data for f in flags],
                            7, rank, world, 2, 2, None, 1)
    for g in gathered:
        assert np.array_equal(g, want)
    assert flags[0][1] == 7 and flags[1][0] == 7
    # argument checks: rows that are not 16-byte multiples cannot be pushed
    odd = np.zeros((2, 7001), np.float32)
    with pytest.raises(_cabi.GateError):
        _cabi.peer_push(lib, odd.ctypes.data, [gathered[0].ctypes.data], 2, 7001 * 4, 7001 * 4, 7001 * 4, 1, None)


def test_get_traces_subranges_on_simulator(lib, monkeypatch):
    """SpectralGate.get_traces(start_frame, end_frame) runs only the reference's units (base.py:167-226):
    a chunk sub-range of the grid (host rows -> slab pipeline; int16 -> staged window), and the single
    padded chunk [0, end) whose right padding is real signal."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    from noisereduce_b200.spectralgate.nonstationary import SpectralGateNonStationary
    y = synth_small(C=2, n=11000)
    kw = dict(chunk_size=3000, padding=400)
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, clip_noise_stationary=True, n_fft=1024, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500, time_mask_smooth_ms=50,
                tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1, **kw)
    cfg = O.GateConfig(sr=SR, stationary=True, **kw)
    sg = SpectralGateStationary(y=y, sr=SR, **args)
    for a, b in ((3500, 8200), (0, 11000), (6000, 9001)):
        out = sg.get_traces(a, b)
        ref = O.reduce_noise(y, SR, cfg=cfg, start_frame=a, end_frame=b)
        assert out.shape == ref.shape == (2, b - a)
        assert P.relinf(out, ref) < P.OUT_TOL
        assert sg._gate.stats()["units"] == 2 * (int((b - 1) / 3000) - int(a / 3000) + 1)
    out = sg.get_traces(1000, 3500)                                    # base.py:222: [0, 3500), one unit per channel
    ref = O.reduce_noise(y, SR, cfg=cfg, start_frame=1000, end_frame=3500)
    assert out.shape == ref.shape == (2, 3500) and P.relinf(out, ref) < P.OUT_TOL
    assert sg._gate.stats()["units"] == 2
    full = sg.get_traces()                                             # the range does not stick
    assert P.relinf(full, O.reduce_noise(y, SR, cfg=cfg)) < P.OUT_TOL
    with pytest.raises(ValueError):
        sg.get_traces(0, 12000)
    # int16 rows, non-stationary gate: staged-window path
    yi = np.round(y * 20000).astype(np.int16)
    a2 = dict(args)
    for k in ("y_noise", "n_std_thresh_stationary", "clip_noise_stationary"):
        a2.pop(k)
    a2.update(time_constant_s=0.3, thresh_n_mult_nonstationary=2, sigmoid_slope_nonstationary=10)
    sn = SpectralGateNonStationary(y=yi, sr=SR, **a2)
    cfgn = O.GateConfig(sr=SR, stationary=False, time_constant_s=0.3, **kw)
    out = sn.get_traces(3100, 9500)
    ref = O.reduce_noise(yi, SR, cfg=cfgn, start_frame=3100, end_frame=9500)
    assert out.dtype == np.int16 and np.max(np.abs(out.astype(np.int64) - ref.astype(np.int64))) <= 1
    out = sn.get_traces(None, 2000)
    ref = O.reduce_noise(yi, SR, cfg=cfgn, end_frame=2000)
    assert out.shape == (2, 2000) and np.max(np.abs(out.astype(np.int64) - ref.astype(np.int64))) <= 1
    # "device" rows (the simulator's device memory is host memory): nothing outside the range is written
    gate = sg._gate
    yc = np.ascontiguousarray(y)
    o = np.full_like(yc, 7.0)
    gate.set_range(1, 1, 2)
    gate.run_device(yc.ctypes.data, o.ctypes.data, np.float32, 2, 11000, 11000, 11000)
    gate.set_range(0)
    assert np.all(o[:, :3000] == 7.0) and np.all(o[:, 9000:] == 7.0)
    assert P.relinf(o[:, 3000:9000], O.reduce_noise(y, SR, cfg=cfg)[:, 3000:9000]) < P.OUT_TOL
    with pytest.raises(_cabi.GateError, match="chunk range"):
        gate.set_range(1, 2, 4)
        gate.run_device(yc.ctypes.data, o.ctypes.data, np.float32, 2, 11000, 11000, 11000)
    gate.set_range(0)


GEN_TOL = 2e-7      # float64 kernels; what is left is the float32 cast of the output / taps


@pytest.mark.parametrize("geo", [
    dict(n_fft=512),
    dict(n_fft=512, win_length=400, hop_length=100),
    dict(n_fft=256, win_length=255, hop_length=50),          # odd window: one more output sample per chunk
    dict(n_fft=128, win_length=100, hop_length=33),          # hop does not divide the window
    dict(n_fft=2048),                                        # stationary 2048 has no tuned kernel
    dict(n_fft=1024, path_flags=4),                          # tuned geometry forced onto the general family
    dict(n_fft=400),                                         # not a power of two: Bluestein through M = 1024
    dict(n_fft=441, win_length=441, hop_length=110),         # odd n_fft: no Nyquist bin
    dict(n_fft=1000, win_length=600, hop_length=150),
], ids=lambda g: "-".join(f"{k}{v}" for k, v in g.items()))
def test_general_geometry_family(lib, geo):
    """Any power-of-two n_fft, win_length <= n_fft, hop_length <= win_length (gate_generic.cuh): every stage
    against the oracle, both gates; decisions bit-exact."""
    geo = dict(geo)
    extra = {k: geo.pop(k) for k in list(geo) if k == "path_flags"}
    y = synth_small(C=2, n=5000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=2000, padding=300, **geo)
    r = P.check_stationary(lib, y, cfg, tap_unit=(1, 1), inject_thresh=False, **extra)
    assert r["thresh_err_db"] < P.THRESH_TOL_DB
    r = P.check_stationary(lib, y, cfg, tap_unit=(2, 0), **extra)
    assert r["mask0_mismatch"] == 0 and r["mask0_on_frac"] > 0.02
    assert r["spec_err"] < GEN_TOL and r["mask_err"] < GEN_TOL and r["out_relinf"] < GEN_TOL
    if "n_fft" in geo and geo["n_fft"] == 2048 and not extra:
        return                                               # non-stationary 2048 is the tuned family (tested above)
    cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=2000, padding=300, time_constant_s=0.2, **geo)
    r = P.check_nonstationary(lib, y, cfg, tap_unit=(1, 1), **extra)
    assert r["spec_err"] < GEN_TOL and r["mask_err"] < GEN_TOL and r["out_relinf"] < GEN_TOL


def test_general_geometry_dtypes_blend_and_ranges(lib, monkeypatch):
    """int16 / float64 rows, prop_decrease < 1, no smoothing, single chunk, sub-ranges -- through reduce_noise()."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    import noisereduce_b200 as nr
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    y = synth_small(C=2, n=6000)
    yi = np.round(y * 20000).astype(np.int16)
    kw = dict(n_fft=256, win_length=200, hop_length=64, chunk_size=2500, padding=300)
    out = nr.reduce_noise(y=yi, sr=SR, stationary=True, prop_decrease=0.7, **kw)
    ref = O.reduce_noise(yi, SR, cfg=O.GateConfig(sr=SR, stationary=True, prop_decrease=0.7, **kw))
    assert out.dtype == np.int16 and np.abs(out.astype(np.int64) - ref.astype(np.int64)).max() <= 1
    y64 = y.astype(np.float64)
    out = nr.reduce_noise(y=y64, sr=SR, stationary=False, prop_decrease=0.6, time_constant_s=0.3, freq_mask_smooth_hz=None,
                          time_mask_smooth_ms=None, **kw)
    ref = O.reduce_noise(y64, SR, cfg=O.GateConfig(sr=SR, stationary=False, prop_decrease=0.6, time_constant_s=0.3,
                                                   freq_mask_smooth_hz=None, time_mask_smooth_ms=None, **kw))
    assert out.dtype == np.float64 and P.relinf(out, ref) < 1e-12            # float64 end to end
    out = nr.reduce_noise(y=y[0], sr=SR, stationary=True, n_fft=512)          # one padded chunk, 1-D input
    ref = O.reduce_noise(y[0], SR, cfg=O.GateConfig(sr=SR, stationary=True, n_fft=512))
    assert out.shape == (6000,) and P.relinf(out, ref) < GEN_TOL
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, clip_noise_stationary=True, n_fft=512, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500, time_mask_smooth_ms=50,
                tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1, chunk_size=2500, padding=300)
    sg = SpectralGateStationary(y=y, sr=SR, **args)
    cfg = O.GateConfig(sr=SR, stationary=True, n_fft=512, chunk_size=2500, padding=300)
    assert P.relinf(sg.get_traces(2600, 5900), O.reduce_noise(y, SR, cfg=cfg, start_frame=2600, end_frame=5900)) < GEN_TOL
    assert P.relinf(sg.get_traces(100, 2000), O.reduce_noise(y, SR, cfg=cfg, start_frame=100, end_frame=2000)) < GEN_TOL


def test_operator_attributes_of_the_reference(lib, monkeypatch):
    """Attributes user code reads off the reference's operator objects (base.py:54-97, stationary.py:47-81)."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    from noisereduce_b200.spectralgate.stationary import SpectralGateStationary
    y = synth_small(C=2, n=6000)
    sg = SpectralGateStationary(y=y, sr=SR, y_noise=None, n_std_thresh_stationary=1.5, chunk_size=2500,
                                clip_noise_stationary=True, padding=400, n_fft=1024, win_length=None, hop_length=None,
                                time_constant_s=2.0, freq_mask_smooth_hz=500, time_mask_smooth_ms=50, tmp_folder=None,
                                prop_decrease=1.0, use_tqdm=False, n_jobs=1)
    assert (sg.n_channels, sg.n_frames, sg.flat, sg.smooth_mask) == (2, 6000, False, True)
    assert (sg._n_fft, sg._win_length, sg._hop_length) == (1024, 1024, 256)
    assert sg._smoothing_filter.shape == (2 * 16 + 1, 2 * 3 + 1) and abs(sg._smoothing_filter.sum() - 1) < 1e-12
    assert np.allclose(sg._smoothing_filter, O.smoothing_filter(16, 3), atol=1e-15)
    yn = sg.y_noise
    assert yn.dtype == np.float32 and yn.shape == (2500,) and np.array_equal(yn, np.mean(y[:, :2500], axis=0))
    info = {}
    O.reduce_noise(y, SR, cfg=O.GateConfig(sr=SR, stationary=True, chunk_size=2500, padding=400), info=info)
    assert sg.noise_thresh.shape == sg.mean_freq_noise.shape == sg.std_freq_noise.shape == (513,)
    assert np.abs(sg.noise_thresh - info["thresh"]).max() < P.THRESH_TOL_DB
    assert np.abs(sg.mean_freq_noise - info["noise_mean"]).max() < P.THRESH_TOL_DB


def test_c_abi_argument_and_state_errors(lib):
    """Error behaviour of the C ABI (negative codes + b200gate_last_error), exercised through the binding."""
    base = dict(surface=_cabi.SURFACE_NUMPY, stationary=1, n_fft=1024, win_length=1024, hop_length=256, n_grad_freq=5,
                n_grad_time=3, chunk_size=3000, padding=400, sr=16000.0, prop_decrease=1.0, n_std_thresh=1.5, top_db=80.0,
                clip_noise=1)
    for bad, msg in ((dict(prop_decrease=float("nan")), "prop_decrease"), (dict(padding=-1), "padding"),
                     (dict(prop_decrease=1.5, surface=_cabi.SURFACE_TORCH, chunk_size=0, padding=0), "prop_decrease"),
                     (dict(n_grad_freq=-1), "smoothing extents"), (dict(hop_length=2000), "unsupported STFT geometry"),
                     (dict(win_length=0), "unsupported STFT geometry"), (dict(surface=7), "unknown surface"),
                     (dict(abi_version=99), "ABI version")):
        with pytest.raises(_cabi.GateError, match=msg):
            _cabi.Gate(lib=lib, **{**base, **bad})
    gate = _cabi.Gate(lib=lib, **base)
    y = synth_small(C=2, n=7000)
    with pytest.raises(_cabi.GateError, match="noise_stats first"):
        gate.run_host(y)                                                 # stationary gate without thresholds
    with pytest.raises(_cabi.GateError, match="expected 513 bins"):
        gate.set_noise_threshold(np.zeros(100))
    gate.noise_stats_host(y)
    out = np.empty_like(y)
    with pytest.raises(_cabi.GateError, match="row strides too small"):
        gate._check(lib.dll.b200gate_run(gate._h, y.ctypes.data, out.ctypes.data, 0, 2, 7000, 6000, 7000, 0, None))
    with pytest.raises(_cabi.GateError, match="bad argument"):
        gate._check(lib.dll.b200gate_run(gate._h, y.ctypes.data, out.ctypes.data, 9, 2, 7000, 7000, 7000, 0, None))
    with pytest.raises(_cabi.GateError, match="bad range"):
        gate.set_range(3, 0, 0)
    gate.set_range(2, 8000)
    with pytest.raises(_cabi.GateError, match="beyond the recording"):
        gate.run_host(y)
    gate.set_range(1, 0, 1)
    with pytest.raises(_cabi.GateError, match="shorter than the range"):
        gate._check(lib.dll.b200gate_run(gate._h, y.ctypes.data, out.ctypes.data, 0, 2, 7000, 7000, 3000, 0, None))
    gate.set_range(0)
    assert P.relinf(gate.run_host(y), O.reduce_noise(y, SR, cfg=O.GateConfig(sr=SR, stationary=True, chunk_size=3000, padding=400,
                                                                               freq_mask_smooth_hz=5 * 16000 / 512 + 1,
                                                                               time_mask_smooth_ms=3 * 16 + 1))) < P.OUT_TOL
    gate.close()


def test_oversized_smoothing_filter_runs_on_the_general_family(lib):
    """Default STFT geometry but a smoothing filter beyond the tuned integer kernels (more than 64 taps a side / 16-bit
    numerators): the library routes the call to the float64 general family instead of refusing it."""
    y = synth_small(C=1, n=30000)
    cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=None, padding=2000, time_mask_smooth_ms=1100)      # nt = 68
    r = P.check_stationary(lib, y, cfg)
    assert r["mask0_mismatch"] == 0 and r["mask_err"] < GEN_TOL and r["out_relinf"] < GEN_TOL
    cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=None, padding=2000, freq_mask_smooth_hz=2100, time_constant_s=0.3)  # nf = 67
    r = P.check_nonstationary(lib, y, cfg)
    assert r["mask_err"] < GEN_TOL and r["out_relinf"] < GEN_TOL


def test_prop_decrease_outside_unit_interval_like_the_reference(lib):
    """reduce_noise() does not validate prop_decrease (stationary.py:108-110): over-subtraction (> 1) and
    negative values are plain arithmetic on the mask."""
    y = synth_small(C=1, n=7000)
    for p_ in (1.4, -0.3):
        cfg = O.GateConfig(sr=SR, stationary=True, chunk_size=3000, padding=400, prop_decrease=p_)
        r = P.check_stationary(lib, y, cfg, tap_unit=(1, 0))
        assert r["mask0_mismatch"] == 0 and r["mask_err"] < 2 * P.MASK_TOL and r["out_relinf"] < 2 * P.OUT_TOL_TIGHT
        cfg = O.GateConfig(sr=SR, stationary=False, chunk_size=3000, padding=400, prop_decrease=p_, time_constant_s=0.3)
        r = P.check_nonstationary(lib, y, cfg, tap_unit=(1, 0))
        assert r["mask_err"] < 2 * P.MASK_TOL_NONSTAT and r["out_relinf"] < 10 * P.OUT_TOL_TIGHT


def test_reference_test_suite_scenarios_on_simulator(lib, monkeypatch, golden_dir):
    """test_reduction.py:6-56 of the reference (its four numpy-path scenarios) on the first 50000 samples of its asset."""
    monkeypatch.setattr(_cabi, "_LIB", lib)
    import noisereduce_b200 as nr
    f = golden.load(golden_dir, "fish_cfg1")
    sr = int(f["sr"])
    for name, y, kw in P.reference_test_suite_scenarios(f["y"], sr, n=50000):
        if name == "stationary_without_noise_clip":
            continue                                   # same kernels as the first scenario; keeps the CPU suite short
        out = nr.reduce_noise(y=y, sr=sr, **kw)
        cfg_kw = {k: v for k, v in kw.items() if k != "y_noise"}
        ref = O.reduce_noise(y, sr, y_noise=kw.get("y_noise"), cfg=O.GateConfig(sr=sr, **cfg_kw))
        assert out.dtype == np.float64 and out.shape == y.shape, name
        assert P.relinf(out, ref) < (P.OUT_TOL_TIGHT if kw["stationary"] else 10 * P.OUT_TOL_TIGHT), name
