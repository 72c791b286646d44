"""The interval form of the mel projection (sygplan::build_mel_intervals, DESIGN.md 4.1b) must actually RUN for the BASELINE filter
banks.  Its planner refuses banks it cannot represent and the launcher then falls back to the tap sweeps -- silently.  That is what
happened to the 44.1 kHz / 2048 / 128-mel bank (BASELINE cfg4) for most of round 2: 7.7e-18 of rounding dust as the weight of the
Nyquist bin in the last filter made the planner refuse, and an A/B of the two forms compared the sweep with itself.  These tests pin
the form through ``syg_debug_last_mel_form`` and check its rows against the oracle (reference: librosa.filters.mel behind
sygnals/core/features/manager.py:205-227)."""
import numpy as np
import pytest

from backends import BACKENDS, get_engine
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth
from test_parity_cabi import check_rows, oracle_rows

BANKS = [  # (sr, n_fft, hop, n_mels, clip length): cfg4 / cfg1 / cfg3 banks of BASELINE.json + the reference's defaults at 1024
    (44100, 2048, 512, 128, 6000), (22050, 2048, 512, 128, 6000), (16000, 512, 160, 40, 3000), (22050, 1024, 256, 64, 5000)]


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


@pytest.mark.parametrize("sr,n_fft,hop,n_mels,L", BANKS)
def test_interval_form_runs_and_matches_the_oracle(eng, sr, n_fft, hop, n_mels, L):
    y = np.stack([synth.long_signal(L, sr, seed=7 + c).astype(np.float32) for c in range(2)])
    fp = {"mfcc": {"n_mels": n_mels}}
    feats = ["mfcc", "rms_energy"]
    p = _ffi.make_params(eng.lib, sr, feats, n_fft, hop, feature_params=fp)
    out = eng.features_host(y.ravel(), eng.units_clips(y.shape[0], y.shape[1]), p)
    assert eng.lib.dll.syg_debug_last_mel_form() == 1, "the interval-form plan was refused: the tap sweeps ran instead"
    for c in range(y.shape[0]):
        names, ref = oracle_rows(y[c], sr, feats, n_fft, hop, fp)
        check_rows(names, out[c], ref)


def test_nyquist_weight_of_the_last_filter_is_applied(eng):
    """A pure Nyquist tone: the only energy sits in the bin the lanes do not own; the last filter sees it through the plan's extra
    weight exactly as the tap sweep does."""
    sr, n_fft, hop, n_mels = 44100, 2048, 512, 128
    n = 8192
    y = (1000.0 * np.cos(np.pi * np.arange(n))).astype(np.float32)[None, :]
    fp = {"mfcc": {"n_mels": n_mels}}
    p = _ffi.make_params(eng.lib, sr, ["mfcc"], n_fft, hop, feature_params=fp)
    out = eng.features_host(y.ravel(), eng.units_clips(1, n), p)
    assert eng.lib.dll.syg_debug_last_mel_form() == 1
    names, ref = oracle_rows(y[0], sr, ["mfcc"], n_fft, hop, fp)
    check_rows(names, out[0], ref)


def test_layout_specialised_kernel_equals_the_plan_specialised_one(eng):
    """BASELINE cfg4's request in the reference's column order runs on Spec44kL (feature set + rows as compile-time constants); the
    same features in another order miss its layout and run on Spec44k.  Same arithmetic: the rows must agree bit for bit."""
    sr, n_fft, hop, L = 44100, 2048, 512, 9000
    y = np.stack([synth.long_signal(L, sr, seed=31 + c).astype(np.float32) for c in range(2)])
    order_l = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]
    order_p = ["rms_energy", "mfcc", "crest_factor", "spectral_contrast", "spectral_rolloff", "spectral_centroid"]
    from sygnals_b200.batch import feature_row_names
    u = eng.units_clips(y.shape[0], y.shape[1])
    out_l = eng.features_host(y.ravel(), u, _ffi.make_params(eng.lib, sr, order_l, n_fft, hop))
    assert eng.lib.dll.syg_debug_last_feature_kernel() == _ffi.FK_SPEC44KL
    out_p = eng.features_host(y.ravel(), u, _ffi.make_params(eng.lib, sr, order_p, n_fft, hop))
    assert eng.lib.dll.syg_debug_last_feature_kernel() == _ffi.FK_SPEC44K
    names_l, names_p = feature_row_names(order_l, None), feature_row_names(order_p, None)
    assert sorted(names_l) == sorted(names_p) and len(names_l) == 24
    for i, n in enumerate(names_l):
        assert np.array_equal(out_l[:, i], out_p[:, names_p.index(n)]), n
    for c in range(y.shape[0]):
        names, ref = oracle_rows(y[c], sr, order_l, n_fft, hop)
        check_rows(names, out_l[c], ref, bin_hz=sr / n_fft, nyq=sr / 2)
