"""Matrix-level entry points of the boundary: mfcc(S=log-mel) (sygnals/core/features/cepstral.py:94-117) and
spectral_contrast(S=|X|) (sygnals/core/features/frequency_domain.py:147-212) through the C ABI against the oracle
(scipy.fftpack.dct as librosa calls it; the shim's spectral_contrast, pinned independently in test_oracle_independent.py)."""
import numpy as np
import pytest
import scipy.fftpack

from backends import BACKENDS, get_engine
from oracle import librosa_shim as shim


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


def _dev(eng, *arrays):
    if getattr(eng, "test_backend", None) == "emu":
        hold = [np.ascontiguousarray(a) for a in arrays]
        return hold, [h.ctypes.data for h in hold]
    import torch
    hold = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]
    return hold, [h.data_ptr() for h in hold]


def _host(h):
    if isinstance(h, np.ndarray):
        return h
    import torch
    torch.cuda.synchronize()
    return h.cpu().numpy()


@pytest.mark.parametrize("n_mels,T,n_mfcc,dct_type,norm,lifter,units", [(128, 173, 13, 2, "ortho", 0.0, 1), (40, 101, 13, 2, "ortho", 22.0, 3),
                                                                       (31, 7, 31, 3, "ortho", 0.0, 2), (64, 50, 20, 2, None, 0.0, 1),
                                                                       (24, 1, 5, 3, None, 10.0, 1)])
def test_mfcc_from_logmel(eng, n_mels, T, n_mfcc, dct_type, norm, lifter, units):
    rng = np.random.default_rng(n_mels + T)
    S = -80.0 * rng.random((units, n_mels, T))                                   # log-power mel values in [-80, 0] dB
    ref = scipy.fftpack.dct(S, axis=-2, type=dct_type, norm=norm)[:, :n_mfcc, :]
    if lifter > 0:
        ref = ref * (1 + (lifter / 2) * np.sin(np.pi * np.arange(1, 1 + n_mfcc) / lifter))[None, :, None]
    out = np.zeros((units, n_mfcc, T), dtype=np.float64)
    hold, (ps, po) = _dev(eng, S, out)
    eng.mfcc_from_logmel_dev(ps, units, n_mels, T, n_mfcc, dct_type, norm == "ortho", lifter, po)
    np.testing.assert_allclose(_host(hold[1]), ref, rtol=1e-12, atol=1e-10)
    # the shim's mfcc(S=...) (what the unmodified reference calls) agrees
    np.testing.assert_allclose(shim.feature.mfcc(S=S[0], n_mfcc=n_mfcc, dct_type=dct_type, norm=norm, lifter=lifter), ref[0], rtol=1e-12, atol=1e-10)


@pytest.mark.parametrize("sr,n_fft,T,n_bands,fmin,q", [(44100, 2048, 37, 6, 200.0, 0.02), (22050, 2048, 20, 6, 200.0, 0.02), (16000, 512, 64, 4, 100.0, 0.1),
                                                       (8000, 256, 5, 3, 300.0, 0.5), (48000, 8192, 6, 6, 200.0, 0.02)])
def test_spectral_contrast_from_magnitudes(eng, sr, n_fft, T, n_bands, fmin, q):
    """No FFT in front of the selection here, so the FP32 engine must meet the 1e-3 dB bar everywhere (no allowance, no mask)."""
    rng = np.random.default_rng(n_fft + T)
    B = 1 + n_fft // 2
    S = (rng.random((B, T)) * 10.0 ** rng.uniform(-5, 1, (B, T))).astype(np.float32)
    S[:, 1] = 0.0                                                                # silent frame
    S[5:40, 2] = S[5, 2]                                                         # ties
    S[:, 3] = np.round(S[:, 3], 1)
    ref = shim.feature.spectral_contrast(S=S.astype(np.float64), sr=sr, n_fft=n_fft, n_bands=n_bands, fmin=fmin, quantile=q)
    out = np.zeros((n_bands + 1, T), dtype=np.float32)
    hold, (ps, po) = _dev(eng, S, out)
    eng.spectral_contrast_from_mag_dev(ps, B, T, sr, n_bands, fmin, q, po)
    got = _host(hold[1]).astype(np.float64)
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() <= 1e-3, np.abs(got - ref).max()


@pytest.mark.parametrize("sr,n_fft,T,n_bands,fmin", [(44100, 128, 9, 6, 200.0), (16000, 64, 40, 6, 200.0), (48000, 512, 3, 4, 50.0)])
def test_spectral_contrast_from_magnitudes_single_bin_band0(eng, sr, n_fft, T, n_bands, fmin):
    """Bin spacing above fmin: band 0 [0, fmin] holds bin 0 only, librosa averages an empty slice for it and power_to_db's top_db
    clamp against the array maximum spreads the NaN: every entry is NaN."""
    rng = np.random.default_rng(n_fft + T)
    B = 1 + n_fft // 2
    S = (rng.random((B, T)) * 10.0 ** rng.uniform(-5, 1, (B, T))).astype(np.float32)
    ref = shim.feature.spectral_contrast(S=S.astype(np.float64), sr=sr, n_fft=n_fft, n_bands=n_bands, fmin=fmin)
    assert ref.shape == (n_bands + 1, T) and np.isnan(ref).all()
    out = np.zeros((n_bands + 1, T), dtype=np.float32)
    hold, (ps, po) = _dev(eng, S, out)
    eng.spectral_contrast_from_mag_dev(ps, B, T, sr, n_bands, fmin, 0.02, po)
    assert np.isnan(_host(hold[1])).all()


def test_matrix_forms_argument_errors(eng):
    out = np.zeros(8, dtype=np.float64)
    with pytest.raises(ValueError):
        eng.mfcc_from_logmel_dev(out.ctypes.data, 1, 4, 2, 0, 2, True, 0.0, out.ctypes.data)        # n_mfcc < 1
    with pytest.raises(ValueError):
        eng.spectral_contrast_from_mag_dev(out.ctypes.data, 129, 2, 8000.0, 6, 200.0, 0.02, out.ctypes.data)   # band above Nyquist


@pytest.mark.gpu
def test_python_mirrors_on_the_gpu():
    """sygnals_b200.core.features.{cepstral.mfcc, frequency_domain.spectral_contrast}: reference signatures, float64 results."""
    from sygnals_b200.core.features import cepstral, frequency_domain
    rng = np.random.default_rng(4)
    S = -80.0 * rng.random((128, 50))
    m = cepstral.mfcc(S=S, sr=22050, n_mfcc=20)
    assert m.dtype == np.float64 and m.shape == (20, 50)
    np.testing.assert_allclose(m, scipy.fftpack.dct(S, axis=-2, type=2, norm="ortho")[:20], rtol=1e-12, atol=1e-10)
    with pytest.raises(NotImplementedError):
        cepstral.mfcc(y=np.zeros(4096), sr=22050)
    with pytest.raises(ValueError):
        cepstral.mfcc()
    mag = rng.random((1025, 31)) * 10.0 ** rng.uniform(-4, 0, (1025, 31))
    c = frequency_domain.spectral_contrast(mag, 44100)
    assert c.dtype == np.float64 and c.shape == (7, 31)
    assert np.abs(c - shim.feature.spectral_contrast(S=mag, sr=44100)).max() <= 1e-3
    with pytest.raises(ValueError):
        frequency_domain.spectral_contrast(mag[0], 44100)
    with pytest.raises(NotImplementedError):
        frequency_domain.spectral_contrast(mag, 44100, linear=True)
    small = rng.random((65, 12))                                                 # n_fft 128 at 44.1 kHz: band 0 = bin 0 only
    assert np.isnan(shim.feature.spectral_contrast(S=small, sr=44100)).all()
    c = frequency_domain.spectral_contrast(small, 44100)
    assert c.dtype == np.float64 and c.shape == (7, 12) and np.isnan(c).all()
