"""oracle/sygnals_oracle.py == the UNMODIFIED reference on random inputs (the ``*_equals_reference`` tests: live only, they
skip where the reference package is not installed, see ``SYGNALS_REFERENCE_ROOT``); the oracle == a snapshot of its OWN
outputs on the same inputs (the ``*_equals_oracle_snapshot`` tests, tests/golden/oracle_snapshot.npz written by
tests/golden/make_oracle_snapshot.py: a regression guard on the oracle, not evidence that it matches the reference); and
the shim == independent in-image implementations (torch.stft, torchaudio mel, scipy dct)."""
import logging
import warnings

import numpy as np
import pytest

import cases
from oracle import librosa_shim, ref_loader
from oracle import sygnals_oracle as O

needs_ref = pytest.mark.skipif(not ref_loader.reference_available(), reason="the reference sygnals package is not installed")

FEATS = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor",
         "zero_crossing_rate", "spectral_bandwidth", "spectral_flatness", "dominant_frequency", "peak_amplitude",
         "mean_amplitude", "std_dev_amplitude", "skewness", "kurtosis", "signal_entropy"]
EF_CASES = [(22050, 22050, 2048, 512), (16000, 16000, 512, 160), (44100, 30000, 2048, 512),
            (22050, 512, 1024, 256), (22050, 100, 1024, 512), (22050, 5000, 1023, 300)]
EF_PARAMS = {"mfcc": {"n_mels": 64, "n_mfcc": 16, "lifter": 22.0}, "spectral_rolloff": {"roll_percent": 0.9},
             "signal_entropy": {"num_bins": 12}}
SEG_CASES = (dict(segment_length_sec=1.0, overlap_ratio=0.25), dict(segment_length_sec=1.0, overlap_ratio=0.5, pad=False),
             dict(segment_length_sec=0.7, overlap_ratio=0.3, min_segment_length_sec=0.2))
STFT_CASES = (dict(n_fft=512), dict(n_fft=1024, hop_length=100, win_length=600, pad_mode="reflect"), dict(n_fft=256, center=False))
AGG_CASES = ("mean", "std", "median", "min", "max", {"f0": "median", "f3": "max"})
# the snapshot was computed on one CPU; numpy on another may order floating-point sums differently
RTOL = ATOL = 1e-10
checksum = cases.checksum


def ef_input(sr, L, fl, hop):
    rng = np.random.default_rng(L + fl)
    t = np.arange(L) / sr
    y = (0.4 * np.sin(2 * np.pi * 440 * t) + 0.05 * rng.standard_normal(L)).astype(np.float32).astype(np.float64)
    return y, sr, fl, hop


def seg_input():
    return np.random.default_rng(3).standard_normal(5300)


def stft_sample_index(size):
    return np.sort(np.random.default_rng(11).choice(size, min(1024, size), replace=False))


def agg_input():
    rng = np.random.default_rng(5)
    feats = {f"f{i}": rng.standard_normal(300) for i in range(4)}
    feats["f1"][rng.integers(0, 300, 40)] = np.nan
    feats["f2"][50:90] = np.nan
    segs = [(0, 10), (10, 11), (50, 90), (0, 300), (290, 300), (20, 20), (280, 310)]
    return feats, segs


@pytest.fixture(scope="module")
def snapshot():
    return cases.load("oracle_snapshot.npz")


@needs_ref
@pytest.mark.parametrize("sr,L,fl,hop", EF_CASES)
def test_extract_features_equals_reference(sr, L, fl, hop):
    warnings.simplefilter("ignore")
    logging.disable(logging.CRITICAL)
    try:
        ref_loader.load_reference()
        from sygnals.core.features.manager import extract_features
        y, sr, fl, hop = ef_input(sr, L, fl, hop)
        fp = EF_PARAMS
        a = extract_features(y, sr, FEATS, frame_length=fl, hop_length=hop, feature_params=fp,
                             output_format="dict_of_arrays")
        b = O.extract_features(y, sr, FEATS, frame_length=fl, hop_length=hop, feature_params=fp)
        assert list(a) == list(b)
        for k in a:
            np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    finally:
        logging.disable(logging.NOTSET)


@pytest.mark.parametrize("i", range(len(EF_CASES)))
def test_extract_features_equals_oracle_snapshot(snapshot, i):
    warnings.simplefilter("ignore")
    y, sr, fl, hop = ef_input(*EF_CASES[i])
    b = O.extract_features(y, sr, FEATS, frame_length=fl, hop_length=hop, feature_params=EF_PARAMS)
    assert list(b) == [str(n) for n in snapshot[f"ef{i}_names"]]
    rows = snapshot[f"ef{i}_rows"]
    assert rows.shape == (len(b), len(b["time"]))
    for k, ref in zip(b, rows):
        np.testing.assert_allclose(b[k], ref, rtol=RTOL, atol=ATOL, err_msg=k)


@needs_ref
def test_segmentation_and_dsp_equal_reference():
    ref_loader.load_reference()
    from sygnals.core.dsp import compute_stft
    from sygnals.core.segmentation import segment_fixed_length
    y = seg_input()
    for kw in SEG_CASES:
        a, b = segment_fixed_length(y, 1000, **kw), O.segment_fixed_length(y, 1000, **kw)
        assert len(a) == len(b) and all(np.array_equal(p, q) for p, q in zip(a, b))
    for kw in STFT_CASES:
        np.testing.assert_array_equal(compute_stft(y, **kw), O.compute_stft(y, **kw))


def test_segmentation_and_dsp_equal_oracle_snapshot(snapshot):
    y = seg_input()
    for i, kw in enumerate(SEG_CASES):
        b = O.segment_fixed_length(y, 1000, **kw)
        assert [len(s) for s in b] == snapshot[f"seg{i}_lengths"].tolist()
        np.testing.assert_allclose(np.array([checksum(s) for s in b]).reshape(len(b), 3), snapshot[f"seg{i}_checksums"],
                                   rtol=RTOL, atol=ATOL)
    for i, kw in enumerate(STFT_CASES):
        D = O.compute_stft(y, **kw)
        assert D.shape == tuple(snapshot[f"stft{i}_shape"]) and D.dtype == np.complex128
        np.testing.assert_allclose(checksum(np.abs(D)), snapshot[f"stft{i}_checksum"], rtol=RTOL)
        np.testing.assert_allclose(D.ravel()[stft_sample_index(D.size)], snapshot[f"stft{i}_sample"], rtol=RTOL, atol=ATOL)


def test_shim_stft_vs_torch():
    import torch
    rng = np.random.default_rng(0)
    y = rng.standard_normal(6000)
    for n_fft, hop, pm in ((512, 128, "constant"), (2048, 512, "constant"), (1024, 256, "reflect")):
        D = librosa_shim.stft(y, n_fft=n_fft, hop_length=hop, pad_mode=pm)
        T = torch.stft(torch.from_numpy(y), n_fft, hop, window=torch.hann_window(n_fft, periodic=True, dtype=torch.float64),
                       center=True, pad_mode=pm, return_complex=True).numpy()
        assert D.shape == T.shape
        assert np.abs(D - T).max() < 1e-10


def test_shim_mel_vs_torchaudio_and_dct():
    import scipy.fftpack
    import torchaudio
    for sr, n_fft, n_mels in ((22050, 2048, 128), (44100, 2048, 128), (16000, 512, 40)):
        W = librosa_shim.filters.mel(sr=sr, n_fft=n_fft, n_mels=n_mels)
        assert W.dtype == np.float32 and W.shape == (n_mels, n_fft // 2 + 1)
        T = torchaudio.functional.melscale_fbanks(n_fft // 2 + 1, 0.0, sr / 2, n_mels, sr, norm="slaney",
                                                  mel_scale="slaney").numpy().T
        assert np.abs(W - T).max() < 5e-7
        assert (W.sum(axis=1) > 0).all()
    n = 40
    x = np.random.default_rng(1).standard_normal((n, 7))
    k = np.arange(n)[:, None]
    basis = np.sqrt(2.0 / n) * np.cos(np.pi * k * (2 * np.arange(n)[None, :] + 1) / (2 * n))
    basis[0] = 1.0 / np.sqrt(n)
    np.testing.assert_allclose(basis @ x, scipy.fftpack.dct(x, axis=0, type=2, norm="ortho"), atol=1e-12)
    w = librosa_shim.filters.get_window("hann", 512)
    np.testing.assert_allclose(w, 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(512) / 512), atol=1e-15)


def test_shim_power_to_db_semantics():
    S = np.array([[1e-12, 1.0], [1e-3, 10.0]])
    d = librosa_shim.power_to_db(S, ref=np.max)
    assert d.max() == 0.0 and d.min() == -80.0
    assert librosa_shim.power_to_db(np.zeros((2, 2)), ref=np.max).tolist() == [[0.0, 0.0], [0.0, 0.0]]


@needs_ref
def test_segment_aggregation_equals_reference():
    import warnings as w
    ref_loader.load_reference()
    from sygnals.core.ml_utils.formatters import format_feature_vectors_per_segment as ref_fn
    feats, segs = agg_input()
    for agg in AGG_CASES:
        with w.catch_warnings():
            w.simplefilter("ignore")
            a = ref_fn(feats, segs, aggregation=agg, output_format="numpy")
        b = O.format_feature_vectors_per_segment(feats, segs, agg)
        np.testing.assert_array_equal(a, b)


def test_segment_aggregation_equals_oracle_snapshot(snapshot):
    feats, segs = agg_input()
    for i, agg in enumerate(AGG_CASES):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            b = O.format_feature_vectors_per_segment(feats, segs, agg)
        ref = snapshot[f"agg{i}"]
        assert b.shape == ref.shape and np.array_equal(np.isnan(b), np.isnan(ref))
        np.testing.assert_allclose(b, ref, rtol=RTOL, atol=ATOL)
