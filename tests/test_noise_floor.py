"""The FP32 noise floor of every transform path, and the floor-sensitive spectral features on tonal, DC, impulse and near-silent
signals.

The parity tests hold spectra to ``|dP| <= 1e-4 P + 1e-6 max P``: in a quiet bin that admits a magnitude error of 1e-3 of the
frame's peak, four to five decades above what an FP32 FFT does.  Here every frame is measured against what FP32 can do on that very
frame (DESIGN.md 2, "FP32 yardstick"):

* ``X64``: the frame of the float32 samples, windowed and transformed in float64 (framed exactly like the oracle's compute_stft);
* two FP32 yardsticks: the float32 product frame * window, transformed by ``scipy.fft.rfft`` (single precision for float32 input)
  and by CPU ``torch.fft.rfft`` in float32.  Two independent implementations keep a lucky agreement of one of them with float64
  from shrinking the allowance to nothing;
* ``spread_k = max over yardsticks |Y_k - X64_k|`` and ``floor = max(max_k spread_k, 2^-24 ||w x||_2)`` per frame.

A transform path passes when ``max_k |X^_k - X64_k| <= C * floor`` on every frame, C = 8.  A feature row passes when
``|f - f64| <= tol(f) + 4 * spread_f``, where ``tol`` is the parity table (test_parity_cabi.row_tol) and ``spread_f`` is the largest
deviation of the oracle's own feature functions applied to the yardstick spectra: the allowance measures how the frame is
conditioned, not a second implementation.  Each test asserts, through the syg_debug_last_* getters, which kernel ran.
"""
import contextlib

import numpy as np
import pytest
import scipy.fft
import scipy.signal
import torch

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth
from test_parity_cabi import check_rows, oracle_rows, row_tol

EPS32 = 2.0 ** -24
C = 8                   # transform error bound in units of the frame's FP32 floor
K_SPREAD = 4            # feature allowance in units of the yardsticks' spread
SIGNALS = synth.EDGE_KINDS + ("tone_bin", "tone_off", "sideband")
SIDEBAND_DB = -90.0


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


# ------------------------------------------------------------------------------------------------ signals
def tone_bins(n_fft):
    """(bin of the tone, bin of the sideband) for a transform of n_fft points: the sideband sits several bins away, beyond the
    periodic Hann window's leakage of a bin-centred tone (exactly the two neighbouring bins)."""
    k0 = max(2, n_fft // 8 + 1)
    return k0, k0 + min(12, n_fft // 2 - 2 - k0)


def make_signal(kind, n, sr, n_fft):
    t = np.arange(n, dtype=np.float64)
    k0, ks = tone_bins(n_fft)
    if kind in synth.EDGE_KINDS:
        return synth.edge_clip(kind, n, sr)
    if kind == "tone_bin":
        y = 0.5 * np.sin(2 * np.pi * k0 * t / n_fft + 0.3)
    elif kind == "tone_off":
        y = 0.5 * np.sin(2 * np.pi * (k0 + 0.37) * t / n_fft + 0.3)
    elif kind == "sideband":
        y = 0.5 * np.sin(2 * np.pi * k0 * t / n_fft + 0.3) + 0.5 * 10 ** (SIDEBAND_DB / 20) * np.sin(2 * np.pi * ks * t / n_fft + 1.1)
    elif kind == "dc_noise":
        y = 3.0 + 1e-3 * np.random.default_rng(n + n_fft).standard_normal(n)
    else:
        raise ValueError(kind)
    return y.astype(np.float32)


def make_units(kind, L, sr, n_fft):
    """Three units per call, so that tiles straddle units: the signal, the signal at 1e-3 of its level, and the signal reversed.
    16-byte aligned rows (the ring kernel's eligibility rule) when L is a multiple of 4."""
    s = make_signal(kind, L, sr, n_fft)
    rows = [s, (s * np.float32(1e-3)).astype(np.float32), s[::-1]]
    buf = np.empty(3 * L + 4, dtype=np.float32)
    off = (-buf.ctypes.data // 4) % 4
    y = buf[off:off + 3 * L].reshape(3, L)
    y[...] = np.stack(rows)
    return y


# ------------------------------------------------------------------------------------------------ FP32 yardstick
def frame_signal(y, n_fft, hop, center=True, pad_mode="constant"):
    """[n_fft, T] frames exactly as librosa takes them: centred padding of n_fft // 2 (or none), frames at multiples of hop."""
    y = np.asarray(y)
    if center:
        y = np.pad(y, n_fft // 2, mode=pad_mode)
    T = 1 + (len(y) - n_fft) // hop
    return y[np.arange(n_fft)[:, None] + hop * np.arange(T)[None, :]]


def window64(n_fft, win_length=None, name="hann"):
    """periodic scipy window of win_length, centred in n_fft"""
    win_length = n_fft if win_length is None else win_length
    w = scipy.signal.get_window(name, win_length, fftbins=True).astype(np.float64)
    lp = (n_fft - win_length) // 2
    return np.pad(w, (lp, n_fft - win_length - lp))


def transforms(fw32, n=None):
    """X64 and the two FP32 yardsticks of float32 windowed frames [n_fft, T] (transform along axis 0, zero padded to n)"""
    X64 = np.fft.rfft(fw32.astype(np.float64), n=n, axis=0)
    Ys = [scipy.fft.rfft(fw32, n=n, axis=0), torch.fft.rfft(torch.from_numpy(np.ascontiguousarray(fw32)), n=n, dim=0).numpy()]
    assert all(Y.dtype == np.complex64 for Y in Ys), "a yardstick left single precision"
    return X64, [Y.astype(np.complex128) for Y in Ys]


class Yardstick:
    """X64 [B, T], the yardstick spectra, and per frame spread [B, T] and floor [T] of one unit's STFT."""

    def __init__(self, y, n_fft, hop, win_length=None, center=True, pad_mode="constant"):
        fr = frame_signal(np.asarray(y, dtype=np.float32), n_fft, hop, center, pad_mode)
        w = window64(n_fft, win_length)
        fw32 = fr * w.astype(np.float32)[:, None]
        assert fw32.dtype == np.float32
        self.X64 = np.fft.rfft(fr.astype(np.float64) * w[:, None], axis=0)
        _, self.Ys = transforms(fw32)
        self.spread = np.max([np.abs(Y - self.X64) for Y in self.Ys], axis=0)
        self.floor = np.maximum(self.spread.max(axis=0), EPS32 * np.linalg.norm(fr.astype(np.float64) * w[:, None], axis=0))
        t = hop * np.arange(fr.shape[1]) - (n_fft // 2 if center else 0)
        self.interior = (t >= 0) & (t + n_fft <= len(y))             # frames inside the signal, clear of the padding


@contextlib.contextmanager
def oracle_on(spectrum):
    """Make the oracle's STFT return ``spectrum(y, n_fft, hop, win_length, center, pad_mode)``: the oracle's own feature code then
    runs on a yardstick spectrum."""
    lib = orc.librosa
    saved = lib.stft

    def stft(y, *, n_fft=2048, hop_length=None, win_length=None, window="hann", center=True, pad_mode="constant", **_):
        assert window == "hann"
        return spectrum(np.asarray(y, dtype=np.float32), n_fft, hop_length, win_length, center, pad_mode)

    lib.stft = stft
    try:
        yield
    finally:
        lib.stft = saved


def yardstick_rows(y, sr, feats, fl, hop, fp, gain=1.0):
    """Oracle rows on X64 (== the plain oracle) and their largest deviation on the yardstick spectra, the yardsticks' error scaled by
    ``gain`` (X64 + gain (Y - X64)): (names, ref [rows, T], spread [rows, T])."""
    names, ref = oracle_rows(y, sr, feats, fl, hop, fp)
    spread = np.zeros_like(ref)
    for i in range(2):
        def spectrum(x, n, h, wl, c, pm):
            ys = Yardstick(x, n, h, wl, c, pm)
            return ys.X64 + gain * (ys.Ys[i] - ys.X64)
        with oracle_on(spectrum):
            n2, r2 = oracle_rows(y, sr, feats, fl, hop, fp)
        assert n2 == names
        spread = np.maximum(spread, np.abs(np.nan_to_num(r2) - np.nan_to_num(ref)))
    return names, ref, spread


def envelope_rows(y, sr, feats, fl, hop, fp):
    """Oracle rows on the edges of the transform bound, |X64| - C floor (clipped at 0) and |X64| + C floor: (names, deviation
    [rows, T]), the sum of both rows' deviations from the float64 rows.  Spectral contrast is a difference of two order statistics
    in dB; each moves by at most C floor in magnitude when every bin does, so this bounds it for any transform that meets the
    floor bound, however the errors fall."""
    names, ref = oracle_rows(y, sr, feats, fl, hop, fp)
    dev = np.zeros_like(ref)
    for sign in (-1.0, 1.0):
        def spectrum(x, n, h, wl, c, pm):
            ys = Yardstick(x, n, h, wl, c, pm)
            return np.maximum(np.abs(ys.X64) + sign * C * ys.floor, 0.0).astype(np.complex128)
        with oracle_on(spectrum):
            n2, r2 = oracle_rows(y, sr, feats, fl, hop, fp)
        assert n2 == names
        dev += np.abs(np.nan_to_num(r2) - np.nan_to_num(ref))
    return names, dev


def test_yardstick_frames_like_the_oracle():
    """The float64 leg of the yardstick is the oracle's compute_stft to 1e-12: same framing, padding and window."""
    rng = np.random.default_rng(3)
    for n_fft, hop, wl, center, pad in [(512, 128, None, True, "constant"), (1024, 200, 800, True, "reflect"), (441, 110, None, True, "constant"),
                                        (256, 64, 201, False, "constant"), (32, 8, None, True, "constant")]:
        y = rng.standard_normal(3000).astype(np.float32)
        ys = Yardstick(y, n_fft, hop, wl, center, pad)
        ref = orc.compute_stft(y.astype(np.float64), n_fft=n_fft, hop_length=hop, win_length=wl, center=center, pad_mode=pad)
        assert ys.X64.shape == ref.shape
        assert np.abs(ys.X64 - ref).max() <= 1e-12 * np.abs(ref).max()
        assert (ys.spread.max(axis=0) > 0).all() and (ys.floor < 1e-5 * np.abs(ref).max(axis=0)).all()


# ------------------------------------------------------------------------------------------------ 2. transform floor: STFT
def check_floor(got, ys, kind, record, what):
    """got: engine output [B, T] of one unit; returns the largest ratio |X^ - X64| / floor over the frames"""
    X64 = ys.X64
    if kind == _ffi.OUT_COMPLEX:
        err = np.abs(got.astype(np.complex128) - X64)
    elif kind == _ffi.OUT_MAGNITUDE:
        err = np.abs(got.astype(np.float64) - np.abs(X64))
    else:                                                             # |X|^2 formed in FP32: one more rounding relative to |X|
        err = np.maximum(np.abs(np.sqrt(got.astype(np.float64)) - np.abs(X64)) - EPS32 * np.abs(X64), 0.0)
    e = err.max(axis=0)
    fl = ys.floor
    assert (e[fl == 0] == 0).all(), f"{what}: {(e[fl == 0] != 0).sum()} all-zero frames are not exactly zero"
    ratio = np.where(fl > 0, e / np.where(fl > 0, fl, 1.0), 0.0)
    record.append(float(ratio.max()))
    assert ratio.max() <= C, f"{what}: frame {ratio.argmax()} error {ratio.max():.2f} x its FP32 floor {fl[ratio.argmax()]:.3e}"


def check_sideband(got, ys, kind, n_fft, what):
    k0, ks = tone_bins(n_fft)
    ref = np.abs(ys.X64[ks])
    mag = np.abs(got[ks].astype(np.complex128)) if kind != _ffi.OUT_POWER else np.sqrt(got[ks].astype(np.float64))
    keep = ys.interior                                                # the edge frames' leakage of the main tone covers the sideband
    rel = np.abs(mag[keep] - ref[keep]) / ref[keep]
    assert keep.sum() >= 2 and rel.max() <= 1e-2, f"{what}: -90 dB sideband off by {100 * rel.max():.3f} %"


MAG, PW, CX = _ffi.OUT_MAGNITUDE, _ffi.OUT_POWER, _ffi.OUT_COMPLEX
# (name, n_fft, hop, out kinds, expected syg_debug_last_stft_path)
STFT_ARMS = [
    ("ring256", 256, 64, (MAG, PW), 1), ("ring512", 512, 128, (MAG, PW), 1), ("ring1024", 1024, 256, (MAG,), 1),
    ("ring2048", 2048, 512, (MAG, PW), 1),
    ("warp32", 32, 8, (CX, MAG), 2), ("warp128", 128, 31, (CX, PW), 2), ("warp512", 512, 127, (CX, MAG), 2),
    ("warp1024", 1024, 256, (CX,), 2), ("warp2048", 2048, 511, (CX, PW), 2),
    ("cta4096", 4096, 1024, (CX,), 3), ("cta8192", 8192, 2048, (CX,), 3),
    ("subfft4096", 4096, 1024, (MAG, PW), 4), ("subfft8192", 8192, 2048, (MAG,), 4),
    ("mixed400", 400, 100, (CX, MAG), 5), ("mixed1000", 1000, 250, (CX, PW), 5), ("mixed441", 441, 110, (CX, MAG), 5),
]
KIND_NAME = {CX: "complex", MAG: "magnitude", PW: "power"}


@pytest.mark.parametrize("signal", SIGNALS)
@pytest.mark.parametrize("arm", STFT_ARMS, ids=[a[0] for a in STFT_ARMS])
def test_stft_floor(eng, arm, signal, record_property):
    name, n_fft, hop, kinds, path = arm
    sr = 22050
    L = 2 * n_fft + 4 * (n_fft // 8) + 4                              # 16-byte rows; partial rounds
    y = make_units(signal, L, sr, n_fft)
    ratios = []
    for kind in kinds:
        out = eng.stft_host(y.reshape(-1), eng.units_clips(3, L), n_fft, hop, n_fft, 0, True, 0, kind)
        assert eng.lib.dll.syg_debug_last_stft_path() == path, f"{KIND_NAME[kind]}: ran stft path {eng.lib.dll.syg_debug_last_stft_path()}"
        for u in range(3):
            ys = Yardstick(y[u], n_fft, hop)
            assert out[u].shape == ys.X64.shape
            what = f"{KIND_NAME[kind]} unit {u}"
            check_floor(out[u], ys, kind, ratios, what)
            if signal == "sideband" and u != 1:
                check_sideband(out[u], ys, kind, n_fft, what)
    record_property("floor_ratio", max(ratios))


# ------------------------------------------------------------------------------------------------ 2. transform floor: Welch
def welch_yardstick(x, fs, nperseg, noverlap, nfft, detrend, scaling):
    """Per-segment X64 [B, S] and floor [S] of scipy's Welch recipe on float32 samples: the detrend (mean removal) in float64 and
    in each yardstick's float32 arithmetic, the window product in float32; plus the one-sided scale."""
    step = nperseg - noverlap
    S = (len(x) - noverlap) // step
    seg = x[np.arange(nperseg)[:, None] + step * np.arange(S)[None, :]]           # float32 [nperseg, S]
    w = window64(nperseg)
    x64 = seg.astype(np.float64)
    if detrend:
        x64 = x64 - x64.mean(axis=0)
        seg_np = seg - seg.mean(axis=0, dtype=np.float32)
        st = torch.from_numpy(np.ascontiguousarray(seg))
        seg_t = (st - st.mean(dim=0)).numpy()
    else:
        seg_np = seg_t = seg
    w32 = w.astype(np.float32)[:, None]
    X64 = np.fft.rfft(x64 * w[:, None], n=nfft, axis=0)
    Ys = [scipy.fft.rfft(seg_np * w32, n=nfft, axis=0), torch.fft.rfft(torch.from_numpy(np.ascontiguousarray(seg_t * w32)), n=nfft, dim=0).numpy()]
    spread = np.max([np.abs(Y.astype(np.complex128) - X64) for Y in Ys], axis=0)
    floor = np.maximum(spread.max(axis=0), EPS32 * np.linalg.norm(x64 * w[:, None], axis=0))
    scale = 1.0 / (fs * np.sum(w * w)) if scaling == 0 else 1.0 / np.sum(w) ** 2
    one = np.full(X64.shape[0], 2.0)
    one[0] = 1.0
    if nfft % 2 == 0:
        one[-1] = 1.0
    return X64, floor, scale * one


WELCH_ARMS = [  # (name, nperseg, nfft, expected syg_debug_last_welch_path)
    ("warp256", 256, 256, _ffi.WELCH_WARP), ("warp1024", 1024, 1024, _ffi.WELCH_WARP), ("warp512_nfft1024", 512, 1024, _ffi.WELCH_WARP),
    ("cta4096", 4096, 4096, _ffi.WELCH_BLOCK), ("mixed1000", 1000, 1000, _ffi.WELCH_MIXED), ("mixed441", 441, 441, _ffi.WELCH_MIXED),
]


@pytest.mark.parametrize("detrend", [True, False], ids=["detrend", "raw"])
@pytest.mark.parametrize("signal", SIGNALS + ("dc_noise",))
@pytest.mark.parametrize("arm", WELCH_ARMS, ids=[a[0] for a in WELCH_ARMS])
def test_welch_floor(eng, arm, signal, detrend, record_property):
    """PSD error bounded through the same floor: with |X^_s - X64_s| <= C floor_s per segment, the averaged one-sided PSD is off by
    at most scale * mean_s(2 |X64_s| C floor_s + (C floor_s)^2), plus the float32 rounding of the power and of the average."""
    name, nperseg, nfft, path = arm
    fs = 25600
    noverlap = nperseg // 2
    L = 4 * nperseg + 4
    y = make_units(signal, L, fs, nfft)
    psd = eng.psd_welch_host(y.ravel(), eng.units_clips(3, L), fs, 0, nperseg, noverlap, nfft, detrend, 0)
    assert eng.lib.dll.syg_debug_last_welch_path() == path
    ratios = []
    for u in range(3):
        _, ref = orc.compute_psd_welch(y[u].astype(np.float64), fs=fs, nperseg=nperseg, noverlap=noverlap, nfft=nfft,
                                       detrend="constant" if detrend else False)
        X64, floor, scale = welch_yardstick(y[u], fs, nperseg, noverlap, nfft, detrend, 0)
        P64 = (scale[:, None] * np.abs(X64) ** 2).mean(axis=1)
        np.testing.assert_allclose(P64, ref, rtol=1e-9, atol=1e-12 * ref.max())        # the float64 leg is scipy's Welch
        unit = scale * (2 * np.abs(X64) * floor + floor ** 2).mean(axis=1)   # the bound per unit of C, C^2 ~ C for C floor << |X|
        err = np.maximum(np.abs(psd[u] - ref) - 4 * EPS32 * ref, 0.0)
        if not (floor > 0).any():
            assert (psd[u] == 0).all(), f"unit {u}: all-zero segments give a non-zero PSD"
            continue
        ratio = (err / np.maximum(unit, 1e-300)).max()
        ratios.append(float(ratio))
        bound = scale * (2 * np.abs(X64) * C * floor + (C * floor) ** 2).mean(axis=1) + 4 * EPS32 * ref
        bad = np.abs(psd[u] - ref) > bound
        assert not bad.any(), f"unit {u}: {bad.sum()} PSD bins beyond {C} x the FP32 floor, worst at bin {np.argmax(err / np.maximum(unit, 1e-300))} ({ratio:.2f} x)"
        if signal == "sideband" and u != 1:
            _, ks = tone_bins(nfft)
            assert abs(np.sqrt(psd[u][ks] / ref[ks]) - 1.0) <= 1e-2, f"unit {u}: -90 dB sideband off by {100 * abs(np.sqrt(psd[u][ks] / ref[ks]) - 1):.3f} %"
    record_property("floor_ratio", max(ratios, default=0.0))


# ------------------------------------------------------------------------------------------------ 4. features
ALL16 = list(_ffi.FEATURE_IDS)
CFG4 = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]
CFG4_REORDERED = ["rms_energy", "mfcc", "crest_factor", "spectral_contrast", "spectral_rolloff", "spectral_centroid"]
RES_FEATS = ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor", "peak_amplitude", "zero_crossing_rate",
             "skewness", "kurtosis", "signal_entropy"]
TIME_ROWS = {"rms_energy", "crest_factor", "peak_amplitude", "mean_amplitude", "std_dev_amplitude", "zero_crossing_rate", "skewness",
             "kurtosis", "signal_entropy"}


def _mels(n_fft):
    n_mels = 10 if n_fft <= 64 else 20 if n_fft <= 256 else 40
    fp = {"mfcc": {"n_mels": n_mels, "n_mfcc": min(13, n_mels)}}
    if n_fft == 64:       # 22.05 kHz / 64 = 344.5 Hz bins: with fmin 200 band 0 holds bin 0 only and the reference's contrast is NaN
        fp["spectral_contrast"] = {"fmin": 400.0, "n_bands": 5}
    return fp


# (name, sr, n_fft, hop, features, feature_params, expected syg_debug_last_feature_kernel, resident min groups or None)
# The plan-specialised n_fft 2048 kernels serve requests without bandwidth / flatness / dominant frequency / mean / std only, and the
# resident kernel requests without contrast either: there the floor probes are centroid, rolloff, contrast and the MFCCs.
FEATURE_ARMS = [
    *[(f"warp{n}" + ("_fmin400" if n == 64 else ""), 22050, n, n // 4, [f for f in ALL16 if n > 32 or f != "spectral_contrast"],
       _mels(n), _ffi.FK_WARP, None) for n in (32, 64, 128, 256, 512, 1024)],
    ("warpwide2048", 44100, 2048, 512, ALL16, None, _ffi.FK_WARP_WIDE, None),
    ("spec44kl2048", 44100, 2048, 512, CFG4, None, _ffi.FK_SPEC44KL, None),
    ("spec44k2048", 44100, 2048, 512, CFG4_REORDERED, None, _ffi.FK_SPEC44K, None),
    ("spec22k2048", 22050, 2048, 512, CFG4, None, _ffi.FK_SPEC22K, None),
    ("resident512", 16000, 512, 160, RES_FEATS, {"mfcc": {"n_mels": 40}}, _ffi.FK_RESIDENT, 1),
    ("block4096", 44100, 4096, 1024, ALL16, None, _ffi.FK_BLOCK, None),
    ("block8192", 44100, 8192, 2048, ALL16, None, _ffi.FK_BLOCK, None),
    *[(f"mixed{n}", 22050, n, n // 4, ALL16, _mels(n), _ffi.FK_MIXED, None) for n in (400, 1000, 441)],
]


def check_dominant(g, ys, bin_hz, what):
    """Tie-aware: the engine's bin must be a maximum of |X64| up to C FP32 floors; on frames with a clear maximum it is the oracle's."""
    M = np.abs(ys.X64)
    b = np.rint(g / bin_hz).astype(np.int64)
    assert np.allclose(g, b * bin_hz, rtol=1e-6, atol=1e-3), f"{what}: dominant frequency not on a bin"
    T = M.shape[1]
    top = M.max(axis=0)
    assert (M[b, np.arange(T)] >= top - C * ys.floor).all(), f"{what}: dominant bin is not a maximum up to the FP32 floor"
    srt = np.sort(M, axis=0)
    clear = srt[-1] - srt[-2] > 2 * C * ys.floor
    assert np.array_equal(b[clear], M.argmax(axis=0)[clear]), f"{what}: dominant bin differs from the oracle's on a clear maximum"


@pytest.mark.parametrize("signal", SIGNALS)
@pytest.mark.parametrize("arm", FEATURE_ARMS, ids=[a[0] for a in FEATURE_ARMS])
def test_features_floor(eng, arm, signal, record_property):
    name, sr, n_fft, hop, feats, fp, fk, res = arm
    L = 2 * n_fft + 3 * hop + 4
    y = make_units(signal, L, sr, n_fft)
    p = _ffi.make_params(eng.lib, sr, feats, n_fft, hop, feature_params=fp)
    if res is not None:
        eng.lib.dll.syg_debug_set_resident_min_groups(res)
    try:
        out = eng.features_host(y.ravel(), eng.units_clips(3, L), p)
    finally:
        eng.lib.dll.syg_debug_set_resident_min_groups(-1)
    assert eng.lib.dll.syg_debug_last_feature_kernel() == fk, f"ran feature kernel {eng.lib.dll.syg_debug_last_feature_kernel()}"
    if res is not None:
        assert eng.lib.dll.syg_debug_last_features_resident() == 1
    if "mfcc" in feats and n_fft == 2048:
        assert eng.lib.dll.syg_debug_last_mel_form() == 1
    bin_hz, nyq = sr / n_fft, sr / 2
    ratio = 0.0
    for u in range(3):
        names, ref, spread = yardstick_rows(y[u], sr, feats, n_fft, hop, fp)
        _, _, spread_c = yardstick_rows(y[u], sr, feats, n_fft, hop, fp, gain=C)
        if "spectral_contrast" in feats:
            _, env = envelope_rows(y[u], sr, feats, n_fft, hop, fp)
            con = [i for i, n in enumerate(names) if n.startswith("contrast_")]
            spread_c[con] = np.maximum(spread_c[con], env[con])
        got = out[u].astype(np.float64)
        assert got.shape == ref.shape
        ys = Yardstick(y[u], n_fft, hop)
        tnames = [n for n in names if n in TIME_ROWS]
        ti = [names.index(n) for n in tnames]
        check_rows(tnames, got[ti], ref[ti], bin_hz=bin_hz, nyq=nyq)                  # no transform in these rows: the parity bars
        for i, n in enumerate(names):
            if n in TIME_ROWS:
                continue
            what = f"unit {u} {n}"
            if n == "dominant_frequency":
                check_dominant(got[i], ys, bin_hz, what)
                continue
            d = np.abs(got[i] - ref[i])
            tol = row_tol(n, ref[i], bin_hz=bin_hz, nyq=nyq) + np.maximum(K_SPREAD * spread[i], spread_c[i])
            assert np.isfinite(got[i]).all(), f"{what}: not finite"
            bad = d > tol
            assert not bad.any(), (f"{what}: frame {np.argmax(d - tol)} off by {d[bad][0]:.4g} (engine {got[i][bad][0]:.6g}, float64 "
                                   f"{ref[i][bad][0]:.6g}, FP32 spread {spread[i][bad][0]:.3g}, at {C} x {spread_c[i][bad][0]:.3g})")
            if n in ("spectral_flatness", "spectral_bandwidth", "spectral_centroid") and signal in ("dc", "tone_bin"):
                s = spread[i] > 0
                if s.any():
                    ratio = max(ratio, float((d[s] / spread[i][s]).max()))
        if signal == "zeros":                          # exact expectations of all-zero frames (frequency_domain.py, time_domain.py)
            d = dict(zip(names, got))
            for n, v in (("spectral_centroid", 0.0), ("spectral_bandwidth", 0.0), ("spectral_flatness", 0.0), ("dominant_frequency", 0.0),
                         ("rms_energy", 0.0), ("crest_factor", 0.0), ("spectral_rolloff", sr * (n_fft // 2) / n_fft)):
                if n in d:
                    assert (d[n] == np.float32(v)).all(), f"{n} of silence: {np.unique(d[n])}"
    record_property("feature_spread_ratio", ratio)
