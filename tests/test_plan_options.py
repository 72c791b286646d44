"""Request options beyond the default plan against the float64 oracle (oracle/sygnals_oracle.py): mel power, analysis window,
DCT type / norm / lifter, the EXTRA spectral statistics at every transform size, spectral contrast bands, and Welch window /
detrend / scaling.  Each option runs code of its own in the kernels (the powf tap sweep, the window table builders, the
unfolded DCT epilogue, the EXTRA instantiations, the Welch detrend and scaling), so each is compared with the oracle at the
transform sizes that select different kernels.  Tests that claim a kernel path assert the debug getter for it, so a silent
fall-back to another kernel fails instead of passing.

Same tolerances as tests/test_parity_cabi.py.  Every case runs on the CPU fiber emulator (test infrastructure) and, under the
``gpu`` marker, on the B200."""
import numpy as np
import pytest
import scipy.fft

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi
from sygnals_b200.core.features import manager
from sygnals_b200.utils import synth
from test_parity_cabi import check_rows, power_close

WINDOWS = ["hamming", "blackman", "boxcar"]

# (n_fft, hop, sr): every warp tile (32 ... 2048), frame_kernel (4096 / 8192) and the mixed-radix kernel (400 = 2^4 5^2, 1000)
SIZES = {32: (8, 16000), 64: (16, 16000), 128: (32, 16000), 256: (64, 16000), 512: (128, 16000), 1024: (256, 22050),
         2048: (512, 44100), 4096: (1024, 48000), 8192: (2048, 48000), 400: (160, 16000), 1000: (250, 16000)}


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


@pytest.fixture
def resident(eng):
    """the unit-resident kernel (frame_warp_kernel STAGE 5) for any batch with at least one unit group"""
    eng.lib.dll.syg_debug_set_resident_min_groups(1)
    yield eng
    eng.lib.dll.syg_debug_set_resident_min_groups(-1)


def oracle_rows(y, sr, features, fl, hop, feature_params=None, center=True, window="hann"):
    r = orc.extract_features(np.asarray(y, dtype=np.float64), sr, list(features), frame_length=fl, hop_length=hop,
                             center=center, window=window, feature_params=feature_params)
    names = [k for k in r if k != "time"]
    return names, np.stack([r[k] for k in names])


def clip(n_fft, sr, n=None):
    n = 3 * n_fft if n is None else n
    return synth.mixture(n, sr, seed=n_fft + n).astype(np.float32)


def contrast_ok(y, fl, hop, window="hann"):
    """frames without bins below the FP32 noise floor (the mask of test_edge_clips_vs_oracle)"""
    S = np.abs(orc.compute_stft(np.asarray(y, dtype=np.float64), n_fft=fl, hop_length=hop, window=window))
    return S.min(axis=0) >= 1e-5 * S.max(axis=0)


def run_features(eng, y, sr, feats, fl, hop, fp=None, window="hann", n_units=1):
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, window=window, feature_params=fp)
    return eng.features_host(y, eng.units_clips(n_units, len(y) // n_units), p)


# ------------------------------------------------------------------------------------------------ mel power
@pytest.mark.parametrize("n_fft", [64, 128, 256, 512, 1024, 2048, 4096, 8192, 400, 1000])
@pytest.mark.parametrize("power", [1.0, 0.5, 3.0])
def test_mel_power_vs_oracle(eng, power, n_fft):
    """S ** power before the mel projection (manager.py:213-217): the powf tap sweep of every kernel family.  RMS rides along so
    the frame kernel also writes a row that is not mel-derived."""
    hop, sr = SIZES[n_fft]
    y = clip(n_fft, sr)
    feats = ["mfcc", "rms_energy"]
    fp = {"mfcc": {"n_mels": 20 if n_fft <= 256 else 40, "power": power}}
    out = run_features(eng, y, sr, feats, n_fft, hop, fp)
    assert eng.lib.dll.syg_debug_last_mel_form() == 0          # the interval form is for power 2 only: the tap sweep ran
    names, ref = oracle_rows(y, sr, feats, n_fft, hop, fp)
    assert out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref)


@pytest.mark.parametrize("power", [1.0, 3.0])
def test_mel_power_on_the_resident_kernel(resident, power):
    eng = resident
    sr, fl, hop, L, n = 16000, 512, 160, 1600, 6
    y = np.concatenate([synth.mixture(L, sr, seed=40 + c) for c in range(n)]).astype(np.float32)
    fp = {"mfcc": {"n_mels": 40, "power": power}}
    out = run_features(eng, y, sr, ["mfcc"], fl, hop, fp, n_units=n)
    assert eng.lib.dll.syg_debug_last_features_resident() == 1
    assert eng.lib.dll.syg_debug_last_mel_form() == 0
    for c in range(n):
        names, ref = oracle_rows(y[c * L:(c + 1) * L], sr, ["mfcc"], fl, hop, fp)
        check_rows(names, out[c], ref)


def test_mel_power_through_the_manager(eng, monkeypatch):
    """extract_features(feature_params={"mfcc": {"power": 1.0}}) as a plugin user calls it, name for name against the oracle."""
    monkeypatch.setattr(_ffi, "engine", lambda device=None: eng)
    sr, fl, hop = 44100, 2048, 512
    y = clip(fl, sr)
    feats = ["mfcc", "spectral_centroid", "rms_energy"]
    fp = {"mfcc": {"power": 1.0}}
    got = manager.extract_features(y, sr, feats, frame_length=fl, hop_length=hop, feature_params=fp, output_format="dict_of_arrays")
    ref = orc.extract_features(y.astype(np.float64), sr, feats, frame_length=fl, hop_length=hop, feature_params=fp)
    assert list(got) == list(ref)
    np.testing.assert_allclose(got["time"], ref["time"], rtol=0, atol=1e-12)
    names = [k for k in ref if k != "time"]
    check_rows(names, np.stack([got[k] for k in names]), np.stack([ref[k] for k in names]), bin_hz=sr / fl)


# ------------------------------------------------------------------------------------------------ analysis window
@pytest.mark.parametrize("n_fft", [64, 256, 1024, 2048, 4096, 400])
@pytest.mark.parametrize("window", WINDOWS)
def test_window_features_vs_oracle(eng, window, n_fft):
    hop, sr = SIZES[n_fft]
    feats = ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy"]
    y = clip(n_fft, sr)
    if sr > 12800 and n_fft >= 1024:                            # six default bands below Nyquist, each with bins
        feats.append("spectral_contrast")
        y = clip(n_fft, sr, n=48 * hop)                         # contrast's 1e-3 dB bar holds for 99 % of entries: enough of them
    fp = {"mfcc": {"n_mels": 20 if n_fft <= 256 else 40}}
    out = run_features(eng, y, sr, feats, n_fft, hop, fp, window=window)
    names, ref = oracle_rows(y, sr, feats, n_fft, hop, fp, window=window)
    assert out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref, bin_hz=sr / n_fft, contrast_ok=contrast_ok(y, n_fft, hop, window))


# (n_fft, hop, win_length, path of the power output, path of the complex output); 1 ring, 2 warp kernel, 3 CTA-cooperative,
# 4 sub-FFT, 5 mixed radix
STFT_CASES = [(512, 128, 400, 1, 2), (1024, 256, 1024, 1, 2), (64, 16, 50, 2, 2), (256, 101, 200, 2, 2),
              (4096, 1024, 3000, 4, 3), (400, 100, 400, 5, 5), (1000, 250, 800, 5, 5)]


@pytest.mark.parametrize("n_fft,hop,win_length,path_power,path_complex", STFT_CASES)
@pytest.mark.parametrize("window", WINDOWS)
def test_window_stft_vs_oracle(eng, window, n_fft, hop, win_length, path_power, path_complex):
    sr = 16000
    y = synth.mixture(8000, sr, seed=3).astype(np.float32)
    u = eng.units_clips(1, len(y))
    wid = _ffi.WINDOW_IDS[window]
    ref = orc.compute_stft(y.astype(np.float64), n_fft=n_fft, hop_length=hop, win_length=win_length, window=window)
    pw = eng.stft_host(y, u, n_fft, hop, win_length, window=wid, out_kind=_ffi.OUT_POWER)
    assert eng.lib.dll.syg_debug_last_stft_path() == path_power
    assert pw[0].shape == ref.shape
    power_close(pw[0].astype(np.float64), np.abs(ref) ** 2)
    D = eng.stft_host(y, u, n_fft, hop, win_length, window=wid, out_kind=_ffi.OUT_COMPLEX)
    assert eng.lib.dll.syg_debug_last_stft_path() == path_complex
    assert D[0].shape == ref.shape
    scale = np.abs(ref).max(axis=0, keepdims=True)
    assert (np.abs(D[0] - ref) <= 2e-6 * scale + 1e-12).all()


@pytest.mark.parametrize("window", WINDOWS)
def test_window_welch_vs_oracle(eng, window):
    sr = 25600
    y = synth.long_signal(2 * sr, sr, seed=9, block_sec=0.25)
    psd = eng.psd_welch_host(y, eng.units_clips(2, sr), sr, _ffi.WINDOW_IDS[window], 1024, 512, 1024, True, 0)
    for c in range(2):
        _, ref = orc.compute_psd_welch(y[c * sr:(c + 1) * sr].astype(np.float64), fs=sr, window=window, nperseg=1024, noverlap=512, nfft=1024)
        assert psd[c].shape == ref.shape
        assert (np.abs(psd[c] - ref) <= 1e-4 * ref + 2e-6 * ref.max()).all()


# ------------------------------------------------------------------------------------------------ DCT type / norm / lifter
DCT_OPTIONS = [dict(dct_type=t, norm=nm, lifter=lf) for t in (1, 2, 3) for nm in ("ortho", None) for lf in (0.0, 22.0)
               if not (t == 1 and nm == "ortho")] + [dict(n_mels=41, n_mfcc=41), dict(n_mels=41, n_mfcc=41, dct_type=3, norm=None)]


def dct_gain(m):
    """[n_mfcc, 1]: how much the requested DCT (and lifter) scales coefficient k over the orthonormal, unliftered one -- the
    L2 norm of its row.  The MFCC bar (abs 1e-3) is set on the orthonormal scale, where the FP32 error of the log-mel input
    (~1e-5 dB) stays far below it; norm=None multiplies coefficient k by about sqrt(2 n_mels) and a lifter by up to
    1 + lifter / 2, and that error with it.  Orthonormal, unliftered requests have gain 1: their bar is unchanged."""
    n_mels, n_mfcc, lifter = m.get("n_mels", 128), m.get("n_mfcc", 13), m.get("lifter", 0.0)
    D = scipy.fft.dct(np.eye(n_mels), type=m.get("dct_type", 2), norm=m.get("norm", "ortho"), axis=0)[:n_mfcc]
    lift = 1.0 + (lifter / 2.0) * np.sin(np.pi * np.arange(1, n_mfcc + 1) / lifter) if lifter > 0 else np.ones(n_mfcc)
    return np.maximum(1.0, np.abs(lift) * np.linalg.norm(D, axis=1))[:, None]


def _dct_id(o):
    return "-".join(f"{k}{v}" for k, v in o.items())


@pytest.mark.parametrize("opts", DCT_OPTIONS, ids=_dct_id)
def test_dct_options_two_kernel_path(eng, opts):
    """finalize_kernel: folded (type 2) and unfolded (types 1 / 3) DCT, unnormalised, liftered, odd n_mels; n_fft 2048, one long unit."""
    sr, fl, hop = 44100, 2048, 512
    y = clip(fl, sr, n=9000)
    fp = {"mfcc": dict({"n_mels": 40, "n_mfcc": 20}, **opts)}
    out = run_features(eng, y, sr, ["mfcc"], fl, hop, fp)
    assert eng.lib.dll.syg_debug_last_features_resident() == 0
    names, ref = oracle_rows(y, sr, ["mfcc"], fl, hop, fp)
    g = dct_gain(fp["mfcc"])
    check_rows(names, out[0] / g, ref / g)


@pytest.mark.parametrize("opts", DCT_OPTIONS, ids=_dct_id)
def test_dct_options_resident_path(resident, opts):
    """the same options through the resident kernel's STAGE 5 epilogue; n_fft 512, several short units"""
    eng = resident
    sr, fl, hop, L, n = 16000, 512, 160, 1600, 5
    y = np.concatenate([synth.mixture(L, sr, seed=70 + c) for c in range(n)]).astype(np.float32)
    fp = {"mfcc": dict({"n_mels": 40, "n_mfcc": 20}, **opts)}
    u = eng.units_clips(n, L)
    p = _ffi.make_params(eng.lib, sr, ["mfcc"], fl, hop, feature_params=fp)
    out = eng.features_host(y, u, p)
    assert eng.lib.dll.syg_debug_last_features_resident() == 1
    eng.lib.dll.syg_debug_set_resident_min_groups(1 << 30)
    two = eng.features_host(y, u, p)
    assert eng.lib.dll.syg_debug_last_features_resident() == 0
    np.testing.assert_allclose(out, two, rtol=0, atol=2e-5)       # the epilogue is finalize_kernel's arithmetic, summed in the same order
    g = dct_gain(fp["mfcc"])
    for c in range(n):
        names, ref = oracle_rows(y[c * L:(c + 1) * L], sr, ["mfcc"], fl, hop, fp)
        check_rows(names, out[c] / g, ref / g)


def test_dct_type1_ortho_is_refused(eng):
    """the DCT table builder has no orthonormal DCT-I (sygplan::build_dct): the request is refused, never computed as another DCT"""
    y = clip(512, 16000)
    with pytest.raises(ValueError):
        run_features(eng, y, 16000, ["mfcc"], 512, 160, {"mfcc": {"n_mels": 40, "dct_type": 1, "norm": "ortho"}})


# ------------------------------------------------------------------------------------------------ EXTRA statistics, contrast
EXTRA = ["spectral_centroid", "spectral_bandwidth", "spectral_flatness", "dominant_frequency", "peak_amplitude", "mean_amplitude",
         "std_dev_amplitude"]


@pytest.mark.parametrize("n_fft", [32, 64, 256, 512, 2048, 4096, 8192, 400])
def test_extra_features_vs_oracle(eng, n_fft):
    """The EXTRA instantiations of every warp tile, frame_kernel and the mixed-radix kernel.  The centroid is requested before the
    bandwidth so the C-ABI rows line up with the oracle's (which injects a centroid column ahead of a bandwidth that comes first)."""
    hop, sr = SIZES[n_fft]
    y = clip(n_fft, sr)
    out = run_features(eng, y, sr, EXTRA, n_fft, hop)
    names, ref = oracle_rows(y, sr, EXTRA, n_fft, hop)
    assert names == EXTRA and out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref, bin_hz=sr / n_fft)


def test_bandwidth_first_through_the_manager(eng, monkeypatch):
    """The manager injects the centroid column ahead of a bandwidth requested first (manager.py:296-301), as the reference does."""
    monkeypatch.setattr(_ffi, "engine", lambda device=None: eng)
    sr, fl, hop = 22050, 1024, 256
    y = clip(fl, sr)
    feats = ["spectral_bandwidth", "spectral_flatness"]
    got = manager.extract_features(y, sr, feats, frame_length=fl, hop_length=hop, output_format="dict_of_arrays")
    ref = orc.extract_features(y.astype(np.float64), sr, feats, frame_length=fl, hop_length=hop)
    assert list(got) == list(ref) == ["time", "spectral_centroid", "spectral_bandwidth", "spectral_flatness"]
    names = list(ref)[1:]
    check_rows(names, np.stack([got[k] for k in names]), np.stack([ref[k] for k in names]), bin_hz=sr / fl)


@pytest.mark.parametrize("bands", ["default", "custom"])
@pytest.mark.parametrize("n_fft", [512, 4096, 8192, 1000])
def test_contrast_sizes_vs_oracle(eng, n_fft, bands):
    hop, sr = SIZES[n_fft]
    y = clip(n_fft, sr, n=max(3 * n_fft, 6000))
    feats = ["spectral_contrast", "spectral_rolloff"]
    fp = None if bands == "default" else {"spectral_contrast": {"n_bands": 4, "fmin": 300.0, "quantile": 0.05}}
    out = run_features(eng, y, sr, feats, n_fft, hop, fp)
    names, ref = oracle_rows(y, sr, feats, n_fft, hop, fp)
    assert out.shape == (1,) + ref.shape
    check_rows(names, out[0], ref, bin_hz=sr / n_fft, contrast_ok=contrast_ok(y, n_fft, hop))


# ------------------------------------------------------------------------------------------------ Welch
@pytest.fixture(scope="module")
def welch_signal():
    sr = 25600
    return sr, synth.long_signal(2 * sr, sr, seed=9, block_sec=0.25)


@pytest.mark.parametrize("nperseg,noverlap,nfft", [(256, 128, 256), (1024, 512, 2048), (500, 100, 512), (1000, 500, 1000)])
@pytest.mark.parametrize("scaling", ["density", "spectrum"])
@pytest.mark.parametrize("detrend", [True, False])
@pytest.mark.parametrize("window", ["hann"] + WINDOWS)
def test_welch_options_vs_oracle(eng, welch_signal, window, detrend, scaling, nperseg, noverlap, nfft):
    """syg_psd_welch_*: window id x detrend flag x scaling mode, zero-padded segments (nfft > nperseg) and the mixed-radix Welch
    kernel (nperseg = nfft = 1000)."""
    sr, y = welch_signal
    psd = eng.psd_welch_host(y, eng.units_clips(2, sr), sr, _ffi.WINDOW_IDS[window], nperseg, noverlap, nfft, detrend,
                             0 if scaling == "density" else 1)
    for c in range(2):
        _, ref = orc.compute_psd_welch(y[c * sr:(c + 1) * sr].astype(np.float64), fs=sr, window=window, nperseg=nperseg,
                                       noverlap=noverlap, nfft=nfft, detrend="constant" if detrend else False, scaling=scaling)
        assert psd[c].shape == ref.shape
        assert (np.abs(psd[c] - ref) <= 1e-4 * ref + 2e-6 * ref.max()).all(), f"worst {np.abs(psd[c] - ref).max() / ref.max():.3e} of max"
