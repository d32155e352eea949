"""Pin oracle/ against the reference's own outputs (tests/golden/*.npz, made by make_golden.py).

CPU-only.  The bar: integer outputs bit-equal; float outputs within 1e-12 relative (the oracle
restates the same float64 arithmetic; only summation order inside the 2-D smoothing differs).
"""
import numpy as np
import pytest

from oracle import spectral_gate_oracle as O
from oracle import torchgate_oracle as TO
from tests.golden import fixtures as golden
from tests.synth_host import synth_small, synth_torchgate


def relinf(a, b):
    a = np.asarray(a)
    b = np.asarray(b)
    dt = np.complex128 if (np.iscomplexobj(a) or np.iscomplexobj(b)) else np.float64
    a, b = a.astype(dt), b.astype(dt)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


@pytest.fixture(scope="module")
def fish(golden_dir):
    return golden.load(golden_dir, "fish_cfg1")


@pytest.fixture(scope="module")
def small(golden_dir):
    return golden.load(golden_dir, "synth_small")


@pytest.fixture(scope="module")
def tgs(golden_dir):
    return golden.load(golden_dir, "torchgate_small")


def test_dft_primitive_matches_definition():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((5, 256))
    assert relinf(O.rfft(x, 256), O.dft_matrix_rfft(x, 256)) < 1e-13
    # zero-padding at the end when the segment is shorter than n
    assert relinf(O.rfft(x[:, :100], 256), O.dft_matrix_rfft(x[:, :100], 256)) < 1e-13
    X = O.rfft(x, 256)
    assert relinf(O.irfft(X, 256), x) < 1e-13


def test_smoothing_filter_is_integer_rational():
    # taps * (nf+1)^2 (nt+1)^2 are the integers (nf+1-|a|)(nt+1-|b|)  (SURVEY.md A.4)
    for nf, nt in [(5, 9), (10, 4), (16, 3), (5, 8), (1, 3), (4, 1)]:
        f = O.smoothing_filter(nf, nt)
        D = (nf + 1) ** 2 * (nt + 1) ** 2
        a = (nf + 1 - np.abs(np.arange(-nf, nf + 1)))[:, None]
        b = (nt + 1 - np.abs(np.arange(-nt, nt + 1)))[None, :]
        assert np.abs(f * D - a * b).max() < 1e-9
        assert abs(f.sum() - 1) < 1e-14


def test_fish_cfg1_stationary_int16_bit_equal(fish):
    info = {}
    out = O.reduce_noise(fish["y"], int(fish["sr"]), cfg=O.GateConfig(sr=int(fish["sr"]), stationary=True), info=info)
    assert out.dtype == np.int16
    assert np.array_equal(out, fish["out_stationary"])
    assert np.abs(info["thresh"] - fish["thresh"]).max() < 1e-9
    assert (info["n_grad_freq"], info["n_grad_time"]) == (5, 8)     # 11 x 17 filter at 44.1 kHz


def test_fish_cfg1_nonstationary_int16_bit_equal(fish):
    out = O.reduce_noise(fish["y"], int(fish["sr"]), cfg=O.GateConfig(sr=int(fish["sr"]), stationary=False))
    assert np.array_equal(out, fish["out_nonstationary"])


def test_fish_cfg1_float32(fish):
    y = (fish["y"] / 32768).astype(np.float32)
    info = {}
    out = O.reduce_noise(y, int(fish["sr"]), cfg=O.GateConfig(sr=int(fish["sr"]), stationary=True), info=info)
    assert out.dtype == np.float32
    assert relinf(out, fish["out_stationary_f32"]) < 1e-7      # equal up to the final float32 cast
    assert np.abs(info["thresh"] - fish["thresh_f32"]).max() < 1e-9


def test_synth_input_is_reproducible(small, tgs):
    assert np.array_equal(synth_small(), small["y"])
    assert np.array_equal(synth_torchgate(), tgs["x"])


CH = dict(chunk_size=12000, padding=1500)


def test_small_stationary_chunked(small):
    y, sr = small["y"], int(small["sr"])
    info = {}
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=True, **CH), info=info)
    assert relinf(out, small["out_stat_chunked"]) < 1e-7
    assert np.abs(info["thresh"] - small["thresh_stat_chunked"]).max() < 1e-9
    # n_jobs does not change the reference's result
    assert np.array_equal(small["out_stat_chunked"], small["out_stat_njobs2"])
    out64 = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=True, **CH), return_float64=True)
    assert relinf(out64.astype(np.float32), small["out_stat_chunked"]) < 1e-7


def test_small_nonstationary_chunked(small):
    y, sr = small["y"], int(small["sr"])
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=False, **CH))
    assert relinf(out, small["out_nonstat_chunked"]) < 1e-7


def test_small_ynoise_prop_decrease(small):
    y, sr = small["y"], int(small["sr"])
    info = {}
    out = O.reduce_noise(y, sr, y_noise=y[:, 3000:11000],
                         cfg=O.GateConfig(sr=sr, stationary=True, prop_decrease=0.8, **CH), info=info)
    assert relinf(out, small["out_stat_ynoise_p08"]) < 1e-7
    assert np.abs(info["thresh"] - small["thresh_stat_ynoise"]).max() < 1e-9


def test_small_nonstationary_2048_f64(small):
    y, sr = small["y"].astype(np.float64), int(small["sr"])
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=False, n_fft=2048, time_constant_s=0.5,
                                                 prop_decrease=0.9))
    assert out.dtype == np.float64
    assert relinf(out, small["out_nonstat_2048_f64"]) < 1e-12


def test_small_single_chunk_flat_and_nosmooth(small):
    y, sr = small["y"], int(small["sr"])
    out = O.reduce_noise(y[0], sr, cfg=O.GateConfig(sr=sr, stationary=True))
    assert out.shape == (y.shape[1],)
    assert relinf(out, small["out_stat_single_chunk"]) < 1e-7
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=True, freq_mask_smooth_hz=None,
                                                 time_mask_smooth_ms=None, **CH))
    assert relinf(out, small["out_stat_nosmooth"]) < 1e-7


def test_prop_decrease_zero_is_identity(small):
    # notebook 1.0 cells 36-40: prop_decrease=0 returns the input "by eye".  Exactly: the mask is
    # all ones, and the zero-padded smoothing attenuates the lowest/highest n_grad_freq bins and
    # the chunk borders (which the chunk centre never sees).  With smoothing off it is the STFT
    # round trip, i.e. the identity to rounding.
    y, sr = small["y"], int(small["sr"])
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=True, prop_decrease=0.0,
                                                 freq_mask_smooth_hz=None, time_mask_smooth_ms=None, **CH),
                         return_float64=True)
    assert relinf(out, y) < 1e-12
    out = O.reduce_noise(y, sr, cfg=O.GateConfig(sr=sr, stationary=True, prop_decrease=0.0, **CH),
                         return_float64=True)
    assert relinf(out, y) < 0.2          # only the band edges differ


def test_errors_match_reference():
    with pytest.raises(ValueError, match="freq_mask_smooth_hz needs to be at least"):
        O.smoothing_extents(48000, 1024, 256, 50, 50)
    with pytest.raises(ValueError, match="time_mask_smooth_ms needs to be at least"):
        O.smoothing_extents(48000, 1024, 256, 500, 1)
    with pytest.raises(ValueError, match="Waveform must be in shape"):
        O.reduce_noise(np.zeros((2, 2, 100)), 16000)


# ---- TorchGate surface ---------------------------------------------------------------------
# The reference builds its window / smoothing taps in float32 and (stationary) smooths the mask
# in float32 even for float64 input, so the float64 oracle pins it to ~1e-7, not 1e-12.
TG_TOL = 2e-6


def test_torchgate_stationary(tgs):
    x, sr = tgs["x"], int(tgs["sr"])
    out = TO.torchgate_forward(x.astype(np.float64), sr, window=tgs["window"], filt=tgs["filt"])
    assert out.shape == tgs["out_stat_f64"].shape == (3, (x.shape[1] // 256) * 256)
    assert relinf(out, tgs["out_stat_f64"]) < TG_TOL
    assert relinf(out, tgs["out_stat_f32"]) < 20 * TG_TOL
    # default (numpy-built) tables differ from torch's by <= 1 ulp(float32)
    out2 = TO.torchgate_forward(x.astype(np.float64), sr)
    assert relinf(out2, tgs["out_stat_f64"]) < TG_TOL


def test_torchgate_nonstationary(tgs):
    x, sr = tgs["x"], int(tgs["sr"])
    out = TO.torchgate_forward(x.astype(np.float64), sr, nonstationary=True, window=tgs["window"], filt=tgs["filt"])
    assert relinf(out, tgs["out_nonstat_f64"]) < TG_TOL
    assert relinf(out, tgs["out_nonstat_f32"]) < 20 * TG_TOL


def test_torchgate_xn(tgs):
    x, sr = tgs["x"].astype(np.float64), int(tgs["sr"])
    out = TO.torchgate_forward(x, sr, xn=x[:1, :6000], prop_decrease=0.7, window=tgs["window"], filt=tgs["filt"])
    assert relinf(out, tgs["out_stat_xn_p07_f64"]) < TG_TOL
    with pytest.raises(Exception, match="x must be bigger than"):
        TO.torchgate_forward(x[:, :1000], sr)


# ---- the performance-faithful port used for the CPU baseline --------------------------------
def test_ref_port_matches_reference(small, fish):
    from oracle import ref_port
    y, sr = small["y"], int(small["sr"])
    out = ref_port.reduce_noise(y, sr, O.GateConfig(sr=sr, stationary=True, **CH), n_jobs=2)
    assert np.array_equal(out, small["out_stat_chunked"])
    out = ref_port.reduce_noise(y, sr, O.GateConfig(sr=sr, stationary=False, **CH))
    assert np.array_equal(out, small["out_nonstat_chunked"])
    out = ref_port.reduce_noise(fish["y"], int(fish["sr"]), O.GateConfig(sr=int(fish["sr"]), stationary=True))
    assert np.array_equal(out, fish["out_stationary"])


def test_get_traces_subranges_match_reference(golden_dir):
    """SpectralGate.get_traces(start_frame, end_frame) (base.py:167-226): chunk-grid branch, and the
    single padded chunk whose right padding is real signal (base.py:222)."""
    g = golden.load(golden_dir, "synth_traces")
    y = synth_small()
    cfg = O.GateConfig(sr=16000, stationary=True, chunk_size=12000, padding=1500)
    for key, (a, b) in {"chunks_13000_28000": (13000, 28000), "chunks_500_24500": (500, 24500),
                        "single_to_9000": (4000, 9000)}.items():
        out = O.reduce_noise(y, 16000, cfg=cfg, start_frame=a, end_frame=b)
        assert out.shape == g[key].shape, key
        assert np.max(np.abs(out.astype(np.float64) - g[key])) < 1e-6 * np.max(np.abs(g[key])), key
    cfg = O.GateConfig(sr=16000, stationary=True, chunk_size=None, padding=1500)
    out = O.reduce_noise(y, 16000, cfg=cfg, end_frame=29000)
    assert out.shape == g["single_to_29000_nochunk"].shape == (2, 29000)
    assert np.max(np.abs(out.astype(np.float64) - g["single_to_29000_nochunk"])) < 1e-6


GEOMETRY_CASES = {
    "stat_512": (dict(stationary=True, n_fft=512), np.float32),
    "nonstat_512_400_100": (dict(stationary=False, n_fft=512, win_length=400, hop_length=100, time_constant_s=0.5), np.float32),
    "stat_256_255_50_i16": (dict(stationary=True, n_fft=256, win_length=255, hop_length=50, prop_decrease=0.9), np.int16),
    "stat_2048": (dict(stationary=True, n_fft=2048), np.float32),
    "nonstat_1024_hop300_f64": (dict(stationary=False, n_fft=1024, hop_length=300, time_constant_s=0.5), np.float64),
    # n_fft not a power of two
    "stat_400": (dict(stationary=True, n_fft=400), np.float32),
    "nonstat_441_odd": (dict(stationary=False, n_fft=441, time_constant_s=0.5), np.float32),
    "stat_1000_600_150": (dict(stationary=True, n_fft=1000, win_length=600, hop_length=150), np.float32),
}


def geometry_input(dtype):
    y = synth_small()
    if dtype == np.int16:
        return np.round(y * 20000).astype(np.int16)
    return y.astype(dtype)


def test_non_default_stft_geometries_match_reference(golden_dir):
    """n_fft / win_length / hop_length off the defaults (base.py:79-86): odd window, hop not dividing the
    window, zero-padded FFT -- the oracle restates scipy's framing for all of them."""
    g = golden.load(golden_dir, "synth_geometry")
    for key, (kw, dt) in GEOMETRY_CASES.items():
        y = geometry_input(dt)
        cfg = O.GateConfig(sr=16000, chunk_size=12000, padding=1500, **kw)
        out = O.reduce_noise(y, 16000, cfg=cfg)
        assert out.dtype == g[key].dtype and out.shape == g[key].shape, key
        if dt == np.int16:
            assert np.abs(out.astype(np.int64) - g[key].astype(np.int64)).max() <= 1, key
        else:
            assert np.max(np.abs(out.astype(np.float64) - g[key])) < 1e-6 * np.max(np.abs(g[key])), key
    info = {}
    O.reduce_noise(synth_small(), 16000, cfg=O.GateConfig(sr=16000, stationary=True, n_fft=512, chunk_size=12000, padding=1500), info=info)
    assert np.max(np.abs(info["thresh"] - g["thresh_512"])) < 1e-9


NON_POW2_KEYS = ("stat_400", "nonstat_441_odd", "stat_1000_600_150", "stat_400_f64", "nonstat_441_f64")

TG_GEOMETRY_CASES = {
    "stat_512_400_100_f64": (dict(n_fft=512, win_length=400, hop_length=100), None, np.float64),
    "nonstat_512_f64": (dict(nonstationary=True, n_fft=512), None, np.float64),
    "stat_2048_xn_f32": (dict(n_fft=2048, prop_decrease=0.8), (slice(0, 1), slice(0, 6000)), np.float32),
    "stat_400_f64": (dict(n_fft=400), None, np.float64),
    "nonstat_441_f64": (dict(nonstationary=True, n_fft=441), None, np.float64),
}


def test_torchgate_non_default_geometries_match_reference(golden_dir):
    """TorchGate with n_fft / win_length / hop_length off the defaults: window centre-padded to n_fft, pad n_fft/2
    (torch.stft center=True), output (L // hop) * hop (torchgate.py:223-262)."""
    g = golden.load(golden_dir, "torchgate_geometry")
    x = synth_torchgate()[:2, :12000]
    for key, (kw, xn_idx, dt) in TG_GEOMETRY_CASES.items():
        xn = None if xn_idx is None else x[xn_idx].astype(np.float64)
        out = TO.torchgate_forward(x.astype(np.float64), 16000, xn=xn, **kw)
        assert out.shape == g[key].shape, key
        assert relinf(out, g[key]) < (TG_TOL if dt == np.float64 else 20 * TG_TOL), key
    assert np.array_equal(TO.hann_window_f32(400), g["window_400"]) or \
        np.abs(TO.hann_window_f32(400) - g["window_400"]).max() <= 2 ** -23
