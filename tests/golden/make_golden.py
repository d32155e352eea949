"""Generate the golden fixtures in this directory by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference, read-only):

    python tests/golden/make_golden.py

The reference ships no golden vectors of its own (its tests assert nothing, SURVEY.md section 4),
so these outputs -- produced by importing timsainb/noisereduce @ 51c8534 with the numpy / scipy /
torch versions recorded in each file -- are what pins oracle/ (tests/test_oracle_golden.py) and,
through it, the CUDA path.  Nothing here is read at run time on the GPU box except the .npz files.
"""
import os
import sys

import numpy as np

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(HERE, "..", ".."))

import joblib  # noqa: E402
import scipy  # noqa: E402
import torch  # noqa: E402
from scipy.io import wavfile  # noqa: E402

import noisereduce as nr  # noqa: E402  (the reference)
from noisereduce.spectralgate.stationary import SpectralGateStationary  # noqa: E402
from noisereduce.torchgate import TorchGate  # noqa: E402

from tests.golden.fixtures import save  # noqa: E402
from tests.synth_host import synth_small, synth_torchgate  # noqa: E402

VERSIONS = np.array(
    [f"reference=51c8534 v3.0.3 numpy={np.__version__} scipy={scipy.__version__} "
     f"torch={torch.__version__} joblib={joblib.__version__}"]
)


def stationary_thresh(y, sr, **kw):
    """noise_thresh as the reference computes it (stationary.py:66-81)."""
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, chunk_size=600000,
                clip_noise_stationary=True, padding=30000, n_fft=1024, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500,
                time_mask_smooth_ms=50, tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1)
    args.update(kw)
    return SpectralGateStationary(y=y, sr=sr, **args).noise_thresh


def traces(y, sr, start, end, **kw):
    """SpectralGateStationary.get_traces(start_frame, end_frame) (base.py:167-226)."""
    args = dict(y_noise=None, n_std_thresh_stationary=1.5, chunk_size=600000,
                clip_noise_stationary=True, padding=30000, n_fft=1024, win_length=None,
                hop_length=None, time_constant_s=2.0, freq_mask_smooth_hz=500,
                time_mask_smooth_ms=50, tmp_folder=None, prop_decrease=1.0, use_tqdm=False, n_jobs=1)
    args.update(kw)
    return SpectralGateStationary(y=y, sr=sr, **args).get_traces(start, end)


def main():
    # ---- config 1: assets/fish.wav (int16 mono 44.1 kHz), defaults -------------------------
    rate, fish = wavfile.read(os.path.join(REF, "assets", "fish.wav"))
    fish_f32 = (fish / 32768).astype(np.float32)
    save(
        "fish_cfg1",
        versions=VERSIONS, sr=rate, y=fish,
        out_stationary=nr.reduce_noise(y=fish, sr=rate, stationary=True),
        out_nonstationary=nr.reduce_noise(y=fish, sr=rate, stationary=False),
        out_stationary_f32=nr.reduce_noise(y=fish_f32, sr=rate, stationary=True),
        thresh=stationary_thresh(fish, rate),
        thresh_f32=stationary_thresh(fish_f32, rate),
    )

    # ---- small seeded multi-channel, multi-chunk cases --------------------------------------
    sr = 16000
    y = synth_small()                       # float32 [2, 30000]
    kw = dict(chunk_size=12000, padding=1500)
    yn = y[:, 3000:11000]
    save(
        "synth_small",
        versions=VERSIONS, sr=sr, y=y,
        out_stat_chunked=nr.reduce_noise(y=y, sr=sr, stationary=True, **kw),
        thresh_stat_chunked=stationary_thresh(y, sr, **kw),
        out_nonstat_chunked=nr.reduce_noise(y=y, sr=sr, stationary=False, **kw),
        out_stat_ynoise_p08=nr.reduce_noise(y=y, sr=sr, stationary=True, y_noise=yn, prop_decrease=0.8, **kw),
        thresh_stat_ynoise=stationary_thresh(y, sr, y_noise=yn, **kw),
        out_nonstat_2048_f64=nr.reduce_noise(y=y.astype(np.float64), sr=sr, stationary=False, n_fft=2048,
                                             time_constant_s=0.5, prop_decrease=0.9),
        out_stat_njobs2=nr.reduce_noise(y=y, sr=sr, stationary=True, n_jobs=2, **kw),
        out_stat_single_chunk=nr.reduce_noise(y=y[0], sr=sr, stationary=True),
        out_stat_nosmooth=nr.reduce_noise(y=y, sr=sr, stationary=True, freq_mask_smooth_hz=None,
                                          time_mask_smooth_ms=None, **kw),
    )

    # ---- get_traces sub-ranges: chunk-grid branch and the single-padded-chunk branch ----------
    save(
        "synth_traces",
        versions=VERSIONS, sr=sr,
        chunks_13000_28000=traces(y, sr, 13000, 28000, **kw),          # chunks 1..2 of 3, trimmed
        chunks_500_24500=traces(y, sr, 500, 24500, **kw),              # chunks 0..2, end on a chunk edge + 500
        single_to_9000=traces(y, sr, 4000, 9000, **kw),                # base.py:222: [0, 9000), right pad = real samples
        single_to_29000_nochunk=traces(y, sr, None, 29000, chunk_size=None, padding=1500),
    )

    # ---- STFT geometries off the default (general-geometry kernel family) ------------------------
    yi16 = np.round(y * 20000).astype(np.int16)
    save(
        "synth_geometry",
        versions=VERSIONS, sr=sr,
        stat_512=nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=512, **kw),
        thresh_512=stationary_thresh(y, sr, n_fft=512, **kw),
        nonstat_512_400_100=nr.reduce_noise(y=y, sr=sr, stationary=False, n_fft=512, win_length=400, hop_length=100,
                                            time_constant_s=0.5, **kw),
        stat_256_255_50_i16=nr.reduce_noise(y=yi16, sr=sr, stationary=True, n_fft=256, win_length=255, hop_length=50,
                                            prop_decrease=0.9, **kw),
        stat_2048=nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=2048, **kw),
        nonstat_1024_hop300_f64=nr.reduce_noise(y=y.astype(np.float64), sr=sr, stationary=False, n_fft=1024,
                                                hop_length=300, time_constant_s=0.5, **kw),
        # n_fft not a power of two (Bluestein in the general family)
        stat_400=nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=400, **kw),
        thresh_400=stationary_thresh(y, sr, n_fft=400, **kw),
        nonstat_441_odd=nr.reduce_noise(y=y, sr=sr, stationary=False, n_fft=441, time_constant_s=0.5, **kw),
        stat_1000_600_150=nr.reduce_noise(y=y, sr=sr, stationary=True, n_fft=1000, win_length=600, hop_length=150, **kw),
    )

    # ---- TorchGate surface (reference on CPU) ------------------------------------------------
    x = synth_torchgate()                   # float32 [3, 24000]
    xt32 = torch.from_numpy(x)
    xt64 = xt32.double()
    tg_s = TorchGate(sr=sr)
    tg_n = TorchGate(sr=sr, nonstationary=True)
    tg_x = TorchGate(sr=sr, prop_decrease=0.7)
    xn = xt64[:1, :6000]
    save(
        "torchgate_small",
        versions=VERSIONS, sr=sr, x=x,
        window=torch.hann_window(1024).numpy(),
        filt=tg_s.smoothing_filter.numpy()[0, 0],
        out_stat_f64=tg_s(xt64).numpy(),
        out_stat_f32=tg_s(xt32).numpy(),
        out_nonstat_f64=tg_n(xt64).numpy(),
        out_nonstat_f32=tg_n(xt32).numpy(),
        out_stat_xn_p07_f64=tg_x(xt64, xn).numpy(),
    )
    # ---- TorchGate off the default STFT geometry (general family, torch surface) -------------------
    xg = x[:2, :12000]
    xg64 = torch.from_numpy(xg).double()
    save(
        "torchgate_geometry",
        versions=VERSIONS, sr=sr,
        window_400=torch.hann_window(400).numpy(),
        stat_512_400_100_f64=TorchGate(sr=sr, n_fft=512, win_length=400, hop_length=100)(xg64).numpy(),
        nonstat_512_f64=TorchGate(sr=sr, nonstationary=True, n_fft=512)(xg64).numpy(),
        stat_2048_xn_f32=TorchGate(sr=sr, n_fft=2048, prop_decrease=0.8)(torch.from_numpy(xg), torch.from_numpy(xg[:1, :6000])).numpy(),
        stat_400_f64=TorchGate(sr=sr, n_fft=400)(xg64).numpy(),
        nonstat_441_f64=TorchGate(sr=sr, nonstationary=True, n_fft=441)(xg64).numpy(),
    )
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()
