"""Parity of the CUDA kernels (called through the C ABI, include/sygb200.h) against

* the committed golden vectors produced by the UNMODIFIED reference (tests/golden/make_golden.py), and
* the oracle (oracle/sygnals_oracle.py) on seeded inputs, incl. the edge cases the reference's tests cover.

Every test runs twice: on the B200 (``gpu`` marker, the product library) and -- the same kernel sources compiled
for the CPU fiber emulator (tests/emu, test infrastructure only) -- in the GPU-less container.

Tolerances (SURVEY.md section 8(a) note; the engine computes in FP32, the reference in float64):
  frame counts / boundaries / shapes                      exact
  power            |dP| <= 1e-4 * P + 1e-6 * max_bin(P) per frame
  MFCC             abs 1e-3
  centroid         rel 1e-5 + 1e-6 * Nyquist (the FP32 noise floor of empty bins is weighted by their frequency)
  rms / crest      rel 1e-5
  rolloff          exact on >= 99.9 % of frames, never more than one bin off
  contrast (dB)    abs 1e-3 dB on >= 99 % of entries, abs 2e-2 dB everywhere: the valley of a band is its smallest
                   magnitude, whose FP32 FFT error is relative to the frame's LARGEST bin (SURVEY 7.3-5), so deep
                   nulls cannot meet 1e-3 dB in FP32.
"""
import numpy as np
import pytest

import cases
from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


def power_close(P, Pref):
    """P, Pref: [..., B, T]"""
    tol = 1e-4 * Pref + 1e-6 * Pref.max(axis=-2, keepdims=True)
    bad = np.abs(P - Pref) > tol
    assert not bad.any(), f"{bad.sum()} power bins out of tolerance, worst excess {(np.abs(P - Pref) - tol).max():.3e}"


def row_tol(n, r, bin_hz=None, nyq=None):
    """The absolute bar of the table above for row ``n`` against reference values ``r``: everywhere for the continuous rows, the
    one-bin limit for rolloff / dominant frequency and the 2e-2 dB limit for contrast.  None for zero_crossing_rate (exact)."""
    r = np.abs(np.asarray(r, dtype=np.float64))
    if n.startswith("mfcc_"):
        return np.full_like(r, 1e-3)
    if n.startswith("contrast_"):
        return np.full_like(r, 2e-2)
    if n == "spectral_centroid":
        return 1e-5 * r + 1e-6 * (24000.0 if nyq is None else nyq)
    if n in ("rms_energy", "crest_factor", "peak_amplitude", "mean_amplitude", "std_dev_amplitude"):
        return 1e-5 * r + 1e-9
    if n in ("spectral_rolloff", "dominant_frequency"):
        return np.full_like(r, (1.0 + 1e-6) * bin_hz)
    if n in ("skewness", "kurtosis"):
        return 2e-5 * r + 2e-6
    if n == "signal_entropy":
        return np.full_like(r, 1e-6)
    if n == "spectral_bandwidth":
        return 1e-4 * r + 1e-2
    if n == "spectral_flatness":
        return 1e-4 * r + 1e-7
    if n == "zero_crossing_rate":
        return None
    raise AssertionError(f"no tolerance defined for {n}")


def check_rows(names, got, ref, bin_hz=None, nyq=None, contrast_ok=None):
    """got/ref: [rows, T] (or [units, rows, T]) in the order of ``names``."""
    if nyq is None and bin_hz is not None:
        nyq = 24000.0
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape
    if got.ndim == 2:
        got, ref = got[None], ref[None]
    contrast_d = []
    for i, n in enumerate(names):
        g, r = got[:, i], ref[:, i]
        d = np.abs(g - r)
        if n.startswith("mfcc_"):
            assert (d <= row_tol(n, r)).all(), f"{n}: max abs err {d.max():.3e}"
        elif n.startswith("contrast_"):
            assert np.isfinite(g).all()
            if contrast_ok is not None:
                d = d[..., contrast_ok]
            if d.size:
                assert d.max() <= 2e-2, f"{n}: max abs err {d.max():.3e} dB"
            contrast_d.append(d.ravel())
        elif n == "spectral_centroid":
            assert bin_hz is not None
            assert (d <= row_tol(n, r, nyq=nyq)).all(), f"{n}: worst {d.max():.3e}"
        elif n in ("rms_energy", "crest_factor", "peak_amplitude", "mean_amplitude", "std_dev_amplitude"):
            assert (d <= row_tol(n, r)).all(), f"{n}: worst rel {(d / (np.abs(r) + 1e-30)).max():.3e}"
        elif n in ("spectral_rolloff", "dominant_frequency"):
            assert bin_hz is not None
            off = d / bin_hz
            assert off.max() <= 1.0 + 1e-6, f"{n}: off by {off.max():.2f} bins"
            assert (off > 0.5).mean() <= 1e-3, f"{n}: {(off > 0.5).sum()} of {off.size} frames differ"
        elif n == "zero_crossing_rate":
            assert np.array_equal(g, r.astype(np.float32)), f"{n}: differs on {(g != r.astype(np.float32)).sum()} frames"   # counts / frame_length
        else:
            assert (d <= row_tol(n, r)).all(), f"{n}: worst {d.max():.3e}"
    if contrast_d and sum(c.size for c in contrast_d):
        allc = np.concatenate(contrast_d)
        assert (allc > 1e-3).mean() <= 0.01, f"{(allc > 1e-3).sum()} of {allc.size} contrast entries above 1e-3 dB"


def oracle_rows(y, sr, features, fl, hop, feature_params=None, center=True):
    r = orc.extract_features(np.asarray(y, dtype=np.float64), sr, list(features), frame_length=fl, hop_length=hop,
                             center=center, feature_params=feature_params)
    names = [k for k in r if k != "time"]
    return names, (np.stack([r[k] for k in names]) if names else np.zeros((0, len(r["time"]))))


# ------------------------------------------------------------------------------------------------ golden vectors
def test_golden_cfg1_mfcc_rms(eng):
    y, sr = cases.cfg1_input()
    g = cases.load("cfg1_mfcc_rms.npz")
    np.testing.assert_allclose(cases.checksum(y), g["in_checksum"], rtol=1e-12)
    p = _ffi.make_params(eng.lib, sr, ["mfcc", "rms_energy"], 2048, 512, feature_params={"mfcc": {"n_mels": 128, "n_mfcc": 20}})
    out = eng.features_host(y, eng.units_clips(1, len(y)), p)
    assert out.shape == (1, 21, 431) and out.dtype == np.float32
    check_rows([str(n) for n in g["names"]], out[0], g["rows"])


@pytest.mark.parametrize("n_fft", [256, 512, 1024, 2048, 4096, 8192])
def test_golden_cfg2_stft(eng, n_fft):
    y, sr = cases.cfg2_input()
    g = cases.load("cfg2_stft_sweep.npz")
    u = eng.units_clips(y.shape[0], y.shape[1])
    D = eng.stft_host(y.ravel(), u, n_fft, n_fft // 4, n_fft)
    mag = eng.stft_host(y.ravel(), u, n_fft, n_fft // 4, n_fft, out_kind=_ffi.OUT_MAGNITUDE)
    pw = eng.stft_host(y.ravel(), u, n_fft, n_fft // 4, n_fft, out_kind=_ffi.OUT_POWER)
    for c in range(y.shape[0]):
        ref = g[f"D_{n_fft}_{c}"].astype(np.complex128)
        assert D[c].shape == ref.shape == (1 + n_fft // 2, 1 + y.shape[1] // (n_fft // 4))
        scale = np.abs(ref).max(axis=0, keepdims=True)
        assert (np.abs(D[c] - ref) <= 2e-6 * scale + 1e-12).all()
        power_close(pw[c].astype(np.float64), np.abs(ref) ** 2)
        power_close(mag[c].astype(np.float64) ** 2, np.abs(ref) ** 2)


@pytest.mark.parametrize("n_fft,hop,n,L", [(32, 8, 5, 300), (64, 16, 7, 1000), (128, 32, 3, 777), (256, 64, 9, 1601), (512, 128, 11, 3000),
                                           (512, 100, 4, 1234), (1024, 256, 3, 5000)])
def test_stft_real_outputs_ragged_batches_vs_oracle(eng, n_fft, hop, n, L):
    """Magnitude / power output of the small transforms (warp-private tiles of 8 consecutive frames, n_fft <= 512): clip counts and
    frame counts that are not multiples of 8, so tiles straddle clips and the last one is partial."""
    rng = np.random.default_rng(n_fft + L)
    y = rng.standard_normal((n, L)).astype(np.float32)
    u = eng.units_clips(n, L)
    mag = eng.stft_host(y.ravel(), u, n_fft, hop, n_fft, out_kind=_ffi.OUT_MAGNITUDE)
    pw = eng.stft_host(y.ravel(), u, n_fft, hop, n_fft, out_kind=_ffi.OUT_POWER)
    for c in range(n):
        ref = np.abs(orc.compute_stft(y[c].astype(np.float64), n_fft=n_fft, hop_length=hop)) ** 2
        assert mag[c].shape == pw[c].shape == ref.shape == (1 + n_fft // 2, 1 + L // hop)
        power_close(pw[c].astype(np.float64), ref)
        power_close(mag[c].astype(np.float64) ** 2, ref)


def test_golden_cfg2_reflect_and_nocenter(eng):
    y, sr = cases.cfg2_input()
    g = cases.load("cfg2_stft_variants.npz")
    u = eng.units_clips(1, y.shape[1])
    D = eng.stft_host(y[0], u, 1024, 200, 800, pad_mode=_ffi.PAD_IDS["reflect"])
    ref = g["D_reflect_1024_800_200"]
    assert D[0].shape == ref.shape
    assert np.abs(D[0] - ref).max() <= 2e-6 * np.abs(ref).max()
    D = eng.stft_host(y[0], u, 512, 128, 512, center=False)
    ref = g["D_nocenter_512_128"]
    assert D[0].shape == ref.shape
    assert np.abs(D[0] - ref).max() <= 2e-6 * np.abs(ref).max()


def test_golden_cfg3_speech_mfcc(eng):
    y, sr = cases.cfg3_input()
    g = cases.load("cfg3_speech_mfcc.npz")
    p = _ffi.make_params(eng.lib, sr, ["mfcc"], 512, 160, feature_params={"mfcc": {"n_mels": 40}})
    out = eng.features_host(y.ravel(), eng.units_clips(y.shape[0], y.shape[1]), p)
    assert out.shape == g["rows"].shape == (10, 13, 101)
    check_rows([str(n) for n in g["names"]], out, g["rows"])


def test_golden_cfg4_env_sound(eng):
    y, sr = cases.cfg4_input()
    g = cases.load("cfg4_env_sound.npz")
    seg_len, seg_hop, starts, valid = eng.lib.segment_table(len(y), sr, 2.0, 0.5, True, None)
    assert (seg_len, seg_hop, len(starts)) == (int(g["seg_len"]), 44100, int(g["n_segments"]))
    p = _ffi.make_params(eng.lib, sr, cases.CFG4_FEATURES, 2048, 512)
    out = eng.features_host(y, eng.units_clips(len(starts), seg_len, total_len=len(y), stride=seg_hop), p)
    assert out.shape == g["rows"].shape == (8, 24, 173)
    check_rows([str(n) for n in g["names"]], out, g["rows"], bin_hz=sr / 2048)
    # explicit segment table == analytic geometry, bit for bit
    out2 = eng.features_host(y, eng.units_table(starts.ctypes.data, valid.ctypes.data, len(starts), seg_len, len(y)), p)
    assert np.array_equal(out, out2)


def test_golden_cfg5_welch(eng):
    y, sr = cases.cfg5_input()
    g = cases.load("cfg5_machinery_psd.npz")
    u = eng.units_clips(6, sr)
    psd, st = eng.psd_welch_host(y.ravel(), u, sr, 0, 1024, 512, 1024, True, 0, stats=True)
    ref = g["psd"]
    assert psd.shape == ref.shape == (6, 513)
    assert (np.abs(psd - ref) <= 1e-4 * ref + 1e-6 * ref.max(axis=1, keepdims=True)).all()
    np.testing.assert_allclose(st[:, 0], g["rms"], rtol=1e-5)
    np.testing.assert_allclose(st[:, 1], g["crest"], rtol=1e-5)
    pp = eng.psd_welch_host(y[0, :4096], eng.units_clips(1, 4096), sr, 0, 4096, 0, 8192, True, 0)
    ref = g["periodogram_8192"]
    assert (np.abs(pp[0] - ref) <= 1e-4 * ref + 1e-6 * ref.max()).all()
    pp = eng.psd_welch_host(y[1, :sr], eng.units_clips(1, sr), sr, 0, 2048, 1024, 2048, True, 1)
    ref = g["welch_2048_spectrum"]
    assert (np.abs(pp[0] - ref) <= 1e-4 * ref + 1e-6 * ref.max()).all()


# ------------------------------------------------------------------------------------------------ oracle, seeded
@pytest.mark.parametrize("sr,fl,hop,n,features,fp", [
    (16000, 512, 160, 16000, ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"], {"mfcc": {"n_mels": 40}}),
    (22050, 1024, 256, 5000, ["spectral_contrast", "mfcc", "peak_amplitude", "spectral_centroid", "spectral_bandwidth", "spectral_flatness",
                              "dominant_frequency", "mean_amplitude", "std_dev_amplitude"], {"mfcc": {"n_mels": 64, "n_mfcc": 20, "lifter": 22.0}}),
    (44100, 2048, 512, 9000, ["crest_factor", "spectral_contrast", "spectral_rolloff"], {"spectral_rolloff": {"roll_percent": 0.5}}),
    (8000, 256, 64, 3001, ["mfcc", "rms_energy"], {"mfcc": {"n_mels": 20, "n_mfcc": 20, "fmin": 100.0, "fmax": 3500.0}}),
    (16000, 64, 16, 700, ["mfcc", "spectral_centroid"], {"mfcc": {"n_mels": 10, "n_mfcc": 5}}),
    (16000, 32, 8, 300, ["spectral_centroid", "spectral_rolloff", "rms_energy"], None),
    (16000, 128, 32, 1000, ["mfcc", "crest_factor"], {"mfcc": {"n_mels": 16, "dct_type": 3}}),
    (22050, 512, 128, 4100, ["mfcc"], {"mfcc": {"n_mels": 23, "n_mfcc": 23}}),                  # odd n_mels (fold centre term), two DMMA m-tiles per parity
    (22050, 1024, 256, 5000, ["mfcc"], {"mfcc": {"n_mels": 46, "n_mfcc": 40, "dct_type": 3}}),  # unfolded tile, three m-tiles
    (48000, 4096, 1024, 20000, ["mfcc", "spectral_centroid", "rms_energy"], None),
    (48000, 8192, 2048, 30000, ["mfcc", "spectral_rolloff", "crest_factor"], None),
])
def test_features_vs_oracle(eng, sr, fl, hop, n, features, fp):
    y = synth.mixture(n, sr, seed=fl + n)
    names, ref = oracle_rows(y, sr, features, fl, hop, fp)
    p = _ffi.make_params(eng.lib, sr, features, fl, hop, feature_params=fp)
    out = eng.features_host(y, eng.units_clips(1, n), p)
    assert out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref, bin_hz=sr / fl)


@pytest.mark.parametrize("case", ["comb32", "comb32_low", "two_level", "quantile10"])
def test_contrast_selection_stress(eng, case):
    """Spectral-contrast selection when the band's largest bins share a lane of the lane-striped layout (tones 32 bins
    apart), when many bins tie, and with a large quantile (n up to 32 per band)."""
    sr, fl, hop, n = 44100, 2048, 512, 6000
    t = np.arange(n) / sr
    rng = np.random.default_rng(5)
    fp = None
    if case in ("comb32", "comb32_low"):
        k0 = 600 if case == "comb32" else 300                      # bins k0 + 32 i: one lane of the top / second band
        y = 1e-2 * rng.standard_normal(n)
        for i in range(13):
            y += (0.05 + 0.002 * i) * np.sin(2 * np.pi * (k0 + 32 * i) * sr / fl * t + i)
    elif case == "two_level":
        y = np.where((np.arange(n) // 7) % 2 == 0, 0.25, -0.25) + 1e-4 * rng.standard_normal(n)
    else:
        y = 0.3 * rng.standard_normal(n)
        fp = {"spectral_contrast": {"quantile": 0.1, "n_bands": 4, "fmin": 400.0}}
    y = y.astype(np.float32)
    feats = ["spectral_contrast"]
    names, ref = oracle_rows(y, sr, feats, fl, hop, fp)
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    out = eng.features_host(y, eng.units_clips(1, n), p)
    S = np.abs(orc.compute_stft(y.astype(np.float64), n_fft=fl, hop_length=hop))
    ok = (S.min(axis=0) >= 1e-5 * S.max(axis=0))
    check_rows(names, out[0], ref, bin_hz=sr / fl, contrast_ok=ok)


@pytest.mark.parametrize("kind", synth.EDGE_KINDS)
def test_edge_clips_vs_oracle(eng, kind):
    sr, fl, hop, n = 22050, 1024, 256, 6000
    y = synth.edge_clip(kind, n, sr)
    feats = ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor", "spectral_contrast"]
    names, ref = oracle_rows(y, sr, feats, fl, hop, {"mfcc": {"n_mels": 40}})
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params={"mfcc": {"n_mels": 40}})
    out = eng.features_host(y, eng.units_clips(1, n), p)
    # contrast is only comparable on frames without bins below the FP32 noise floor (in the reference those bins hold
    # float64 round-off, here float32 round-off; both are noise, and both sit near the amin=1e-10 clamp)
    S = np.abs(orc.compute_stft(y.astype(np.float64), n_fft=fl, hop_length=hop))
    ok = (S.min(axis=0) >= 1e-5 * S.max(axis=0))          # all-zero frames stay comparable (exactly 0 dB both sides)
    if kind in ("zeros",):
        # all-zero frames: centroid 0, rolloff = freqs[-1], rms 0, crest 0, mfcc of a flat -80 dB... exact expectations
        d = dict(zip(names, out[0]))
        assert (d["spectral_centroid"] == 0).all() and (d["rms_energy"] == 0).all() and (d["crest_factor"] == 0).all()
        assert np.allclose(d["spectral_rolloff"], sr / 2)
    check_rows(names, out[0], ref, bin_hz=sr / fl, contrast_ok=ok)


def test_short_and_ragged_units(eng):
    """Units shorter than a frame (manager test: 512 samples @ frame 1024 -> 3 frames, 100 samples -> 1 frame), a ragged
    tail (zero-padded like segment_fixed_length(pad=True)) and a unit entirely past the end of the buffer."""
    sr, fl, hop = 22050, 1024, 256
    y = synth.mixture(2000, sr, seed=5)
    for n in (512, 100, 1):
        names, ref = oracle_rows(y[:n], sr, ["mfcc", "rms_energy", "crest_factor"], fl, hop)
        p = _ffi.make_params(eng.lib, sr, ["mfcc", "rms_energy", "crest_factor"], fl, hop)
        out = eng.features_host(y[:n], eng.units_clips(1, n), p)
        assert out.shape[2] == 1 + n // hop == ref.shape[1]
        check_rows(names, out[0], ref, bin_hz=sr / fl)
    # ragged: 3 units of 900 samples over a 2000-sample buffer; the third has 200 valid samples, a fourth none
    p = _ffi.make_params(eng.lib, sr, ["rms_energy", "spectral_centroid", "mfcc"], fl, hop)
    out = eng.features_host(y, eng.units_clips(4, 900, total_len=2000, stride=900), p)
    for u in range(4):
        seg = np.zeros(900, dtype=np.float32)
        v = max(0, min(900, 2000 - 900 * u))
        seg[:v] = y[900 * u:900 * u + v]
        names, ref = oracle_rows(seg, sr, ["rms_energy", "spectral_centroid", "mfcc"], fl, hop)
        check_rows(names, out[u], ref, bin_hz=sr / fl)


def test_empty_and_errors(eng):
    p = _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160)
    out = eng.features_host(np.zeros(0, np.float32), eng.units_clips(0, 16000), p)
    assert out.shape == (0, 13, 101)
    # center=False, unit shorter than a frame: zero frames, nothing written
    p2 = _ffi.make_params(eng.lib, 16000, ["rms_energy"], 512, 160, center=False)
    out = eng.features_host(np.zeros(100, np.float32), eng.units_clips(1, 100), p2)
    assert out.shape == (1, 1, 0)
    with pytest.raises(NotImplementedError):
        eng.features_host(np.zeros(4000, np.float32), eng.units_clips(1, 4000), _ffi.make_params(eng.lib, 16000, ["mfcc"], 1006, 160))   # 2 * 503: no kernel for this length
    with pytest.raises(ValueError):
        eng.features_host(np.zeros(4000, np.float32), eng.units_clips(1, 4000),
                          _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160, feature_params={"mfcc": {"n_mfcc": 200}}))
    with pytest.raises(ValueError):   # librosa: "Frequency band exceeds Nyquist" (sr <= 12800 with the default bands)
        eng.features_host(np.zeros(4000, np.float32), eng.units_clips(1, 4000), _ffi.make_params(eng.lib, 8000, ["spectral_contrast"], 512, 160))
    with pytest.raises(ValueError):
        eng.stft_host(np.zeros(4000, np.float32), eng.units_clips(1, 4000), 512, 0, 512)


def test_batch_equals_single_units(eng):
    """Determinism / independence: a unit's rows do not depend on its neighbours in the batch."""
    sr = 16000
    clips = synth.clip_batch(9, 4000, sr, seed=77, edges=False)
    p = _ffi.make_params(eng.lib, sr, ["mfcc", "spectral_contrast", "spectral_rolloff", "rms_energy"], 512, 160, feature_params={"mfcc": {"n_mels": 40}})
    allout = eng.features_host(clips.ravel(), eng.units_clips(9, 4000), p)
    for c in (0, 4, 8):
        one = eng.features_host(clips[c], eng.units_clips(1, 4000), p)
        assert np.array_equal(one[0], allout[c])


def test_welch_vs_oracle_shapes(eng):
    sr = 25600
    y = synth.long_signal(3 * sr, sr, seed=9, block_sec=0.25)
    for nperseg, nov, nfft in ((1024, 512, 1024), (256, 128, 256), (500, 100, 512), (64, 0, 64)):
        u = eng.units_clips(3, sr)
        psd = eng.psd_welch_host(y, u, sr, 0, nperseg, nov, nfft, True, 0)
        for c in range(3):
            f, ref = orc.compute_psd_welch(y[c * sr:(c + 1) * sr].astype(np.float64), fs=sr, nperseg=nperseg, noverlap=nov, nfft=nfft)
            assert psd[c].shape == ref.shape
            assert (np.abs(psd[c] - ref) <= 1e-4 * ref + 2e-6 * ref.max()).all()


def test_pcm16_ingest_equals_float_path(eng):
    """syg_features_host_pcm16: 16-bit PCM widened on the device (x / 32768, libsndfile's normalisation behind librosa.load,
    sygnals/core/audio/io.py:84-95) must give bit-identical rows to the float32 path on the same samples."""
    sr, n = 22050, 30000
    rng = np.random.default_rng(9)
    t = np.arange(n) / sr
    pcm = np.clip(9000 * np.sin(2 * np.pi * 440 * t) + 3000 * rng.standard_normal(n), -32768, 32767).astype(np.int16)
    pcm[:7] = [-32768, 32767, 0, 1, -1, 12345, -12345]
    feats = ["mfcc", "spectral_centroid", "rms_energy", "crest_factor", "spectral_contrast"]
    p = _ffi.make_params(eng.lib, sr, feats, 1024, 256, feature_params={"mfcc": {"n_mels": 40}})
    u = eng.units_clips(3, 10000)
    a = eng.features_host(pcm, u, p)                                  # int16 -> PCM16 entry point
    b = eng.features_host(pcm.astype(np.float32) / np.float32(32768.0), u, p)
    assert a.dtype == np.float32 and np.array_equal(a, b)
    names, ref = oracle_rows(pcm[:10000].astype(np.float64) / 32768.0, sr, feats, 1024, 256, {"mfcc": {"n_mels": 40}})
    check_rows(names, a[0], ref, bin_hz=sr / 1024)


def _dev_buffers(eng, *arrays):
    """'Device' copies of numpy arrays for the engine under test: CUDA tensors on the B200, the arrays themselves on the
    CPU emulator build (whose device memory is host memory).  Returns (holders, pointers)."""
    if getattr(eng, "test_backend", None) == "emu":
        hold = [np.ascontiguousarray(a) for a in arrays]
        return hold, [h.ctypes.data for h in hold]
    import torch
    hold = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]
    return hold, [h.data_ptr() for h in hold]


def _host(eng, h):
    return h if isinstance(h, np.ndarray) else h.cpu().numpy()


@pytest.mark.parametrize("agg", ["mean", "std", "median", "min", "max", "mixed"])
def test_segment_aggregation_vs_oracle(eng, agg):
    """syg_aggregate_f32 == format_feature_vectors_per_segment (formatters.py:51-163): NaN-aware, per-feature methods,
    invalid segments -> NaN rows, odd/even medians, negative values, single-frame segments."""
    rng = np.random.default_rng(12)
    names = [f"f{i}" for i in range(5)]
    N = 400
    feats = {n: (rng.standard_normal(N) * 10.0 ** rng.integers(-2, 3)).astype(np.float32).astype(np.float64) for n in names}
    feats["f1"][rng.integers(0, N, 60)] = np.nan
    feats["f2"][100:140] = np.nan                                    # one segment entirely NaN for this feature
    feats["f3"][:] = np.round(feats["f3"])                           # many ties
    segs = [(0, 1), (1, 3), (3, 36), (36, 100), (100, 140), (140, 141), (150, 400), (0, 400), (390, 400), (50, 50), (380, 420)]
    aggregation = {"f0": "median", "f1": "std", "f2": "max", "f3": "median", "f4": "min"} if agg == "mixed" else agg
    ref = orc.format_feature_vectors_per_segment(feats, segs, aggregation)
    ids = [_ffi.AGG_IDS[aggregation.get(n, "mean") if isinstance(aggregation, dict) else aggregation] for n in names]
    off = np.array([s if (0 <= s < N and s < e <= N) else 0 for s, e in segs], dtype=np.int64)
    ln = np.array([e - s if (0 <= s < N and s < e <= N) else 0 for s, e in segs], dtype=np.int32)
    mat = np.stack([feats[n].astype(np.float32) for n in names])
    out = np.zeros((len(segs), len(names)), dtype=np.float64)
    hold, (pm, po, pl_, pout) = _dev_buffers(eng, mat, off, ln, out)
    eng.aggregate_dev(pm, len(segs), len(names), N, ids, pout, seg_off_ptr=po, seg_len_ptr=pl_)
    if not isinstance(hold[3], np.ndarray):
        import torch
        torch.cuda.synchronize()
    got = _host(eng, hold[3])
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    if agg in ("median", "min", "max"):
        assert np.array_equal(got[ok], ref[ok])                      # selections of float32 values: exact
    else:
        np.testing.assert_allclose(got[ok], ref[ok], rtol=1e-12, atol=1e-12)
    # regular layout [n_seg, rows, T] without tables
    T, n_seg = 37, 9
    cube = rng.standard_normal((n_seg, len(names), T)).astype(np.float32)
    cube[2, 1, 5:9] = np.nan
    out2 = np.zeros((n_seg, len(names)), dtype=np.float64)
    hold2, (pc, pout2) = _dev_buffers(eng, cube, out2)
    eng.aggregate_dev(pc, n_seg, len(names), T, ids, pout2, fixed_len=T)
    if not isinstance(hold2[1], np.ndarray):
        import torch
        torch.cuda.synchronize()
    got2 = _host(eng, hold2[1])
    for s in range(n_seg):
        d = {n: cube[s, j].astype(np.float64) for j, n in enumerate(names)}
        r = orc.format_feature_vectors_per_segment(d, [(0, T)], aggregation)[0]
        np.testing.assert_allclose(got2[s], r, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("sr,fl,hop,n,center", [(22050, 1024, 256, 6000, True), (16000, 512, 160, 3001, True), (44100, 2048, 512, 9000, False),
                                               (8000, 64, 16, 700, True), (48000, 4096, 1024, 20000, True)])
def test_time_extra_features_vs_oracle(eng, sr, fl, hop, n, center):
    """zero_crossing_rate (edge padding), skewness, kurtosis, signal_entropy (time_extra_kernel) alone and mixed with kernel features."""
    y = synth.long_signal(n, sr, seed=fl + n, block_sec=0.05)        # silent, DC and noisy blocks: flat frames, ties at bin edges
    feats = ["zero_crossing_rate", "skewness", "rms_energy", "kurtosis", "signal_entropy", "spectral_centroid"]
    fp = {"signal_entropy": {"num_bins": 12}} if fl == 512 else None
    names, ref = oracle_rows(y, sr, feats, fl, hop, fp, center=center)
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, center=center, feature_params=fp)
    out = eng.features_host(y, eng.units_clips(1, n), p)
    assert out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref, bin_hz=sr / fl)
    only = ["skewness", "zero_crossing_rate"]                        # no frame-kernel feature at all
    names2, ref2 = oracle_rows(y, sr, only, fl, hop, None, center=center)
    out2 = eng.features_host(y, eng.units_clips(1, n), _ffi.make_params(eng.lib, sr, only, fl, hop, center=center))
    check_rows(names2, out2[0], ref2, bin_hz=sr / fl)
    # padded units: the zero tail is part of the unit (zcr's edge value is then 0), three units per call
    u = eng.units_clips(3, n // 2, total_len=n, stride=n // 3)
    out3 = eng.features_host(y, u, p)
    for i in range(3):
        seg = np.zeros(n // 2, dtype=np.float32)
        v = max(0, min(n // 2, n - i * (n // 3)))
        seg[:v] = y[i * (n // 3): i * (n // 3) + v]
        _, r3 = oracle_rows(seg, sr, feats, fl, hop, fp, center=center)
        check_rows(names, out3[i], r3, bin_hz=sr / fl)
