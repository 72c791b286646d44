"""Pins oracle/sygnals_oracle.py against golden vectors produced by the UNMODIFIED reference
(tests/golden/make_golden.py).  Runs on CPU, here and on the GPU box."""
import numpy as np
import pytest

import cases
from oracle import sygnals_oracle as O


def _close(a, b, rtol=1e-9, atol=1e-9):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def test_cfg1_mfcc_rms():
    g = cases.load("cfg1_mfcc_rms.npz")
    y, sr = cases.cfg1_input()
    _close(cases.checksum(y), g["in_checksum"], 1e-12, 0)
    r = O.extract_features(y.astype(np.float64), sr, ["mfcc", "rms_energy"], 2048, 512,
                           feature_params={"mfcc": {"n_mels": 128, "n_mfcc": 20}})
    assert [k for k in r if k != "time"] == [str(n) for n in g["names"]]
    assert len(r["time"]) == 431
    _close(r["time"], g["time"])
    _close(cases.stack_rows(r, g["names"]), g["rows"])


def test_cfg2_stft_sweep():
    g = cases.load("cfg2_stft_sweep.npz")
    clips, sr = cases.cfg2_input()
    _close(cases.checksum(clips), g["in_checksum"], 1e-12, 0)
    for n_fft in (256, 512, 1024, 2048, 4096, 8192):
        for c in range(2):
            D = O.compute_stft(clips[c].astype(np.float64), n_fft=n_fft, hop_length=n_fft // 4)
            G = g[f"D_{n_fft}_{c}"]
            assert D.shape == G.shape == (1 + n_fft // 2, 1 + 8000 // (n_fft // 4))
            assert D.dtype == np.complex128
            scale = np.abs(G).max()
            assert np.abs(D - G).max() <= 2e-7 * scale  # golden stored as complex64
    g = cases.load("cfg2_stft_variants.npz")
    _close(cases.checksum(clips), g["in_checksum"], 1e-12, 0)
    D = O.compute_stft(clips[0].astype(np.float64), n_fft=1024, hop_length=200, win_length=800, pad_mode="reflect")
    assert np.abs(D - g["D_reflect_1024_800_200"]).max() <= 2e-7 * np.abs(D).max()
    D = O.compute_stft(clips[0].astype(np.float64), n_fft=512, hop_length=128, center=False)
    assert D.shape == g["D_nocenter_512_128"].shape
    assert np.abs(D - g["D_nocenter_512_128"]).max() <= 2e-7 * np.abs(D).max()


def test_cfg3_speech_mfcc():
    g = cases.load("cfg3_speech_mfcc.npz")
    clips, sr = cases.cfg3_input()
    _close(cases.checksum(clips), g["in_checksum"], 1e-12, 0)
    for i, c in enumerate(clips):
        r = O.extract_features(c.astype(np.float64), sr, ["mfcc"], 512, 160, feature_params={"mfcc": {"n_mels": 40}})
        assert len(r) == 14 and len(r["time"]) == 101
        _close(cases.stack_rows(r, g["names"]), g["rows"][i])


def test_cfg4_env_sound():
    g = cases.load("cfg4_env_sound.npz")
    y, sr = cases.cfg4_input()
    _close(cases.checksum(y), g["in_checksum"], 1e-12, 0)
    segs = O.segment_fixed_length(y.astype(np.float64), sr, 2.0, overlap_ratio=0.5, pad=True)
    assert len(segs) == int(g["n_segments"]) == 8 and len(segs[0]) == int(g["seg_len"]) == 88200
    np.testing.assert_array_equal(segs[-1][-4:], g["last_segment_tail"])
    for i, s in enumerate(segs):
        r = O.extract_features(s, sr, cases.CFG4_FEATURES, 2048, 512)
        assert [k for k in r if k != "time"] == [str(n) for n in g["names"]]
        assert len(r["time"]) == 173 and len(r) == 25
        _close(cases.stack_rows(r, g["names"]), g["rows"][i], 1e-9, 1e-8)


def test_cfg5_machinery_psd():
    g = cases.load("cfg5_machinery_psd.npz")
    ch, sr = cases.cfg5_input()
    _close(cases.checksum(ch), g["in_checksum"], 1e-12, 0)
    u = 0
    for c in range(3):
        for w in range(2):
            x = ch[c, w * sr:(w + 1) * sr].astype(np.float64)
            f, p = O.compute_psd_welch(x, fs=sr, nperseg=1024, noverlap=512)
            _close(f, g["freqs"])
            _close(p, g["psd"][u], 1e-10, 0)
            f2, p2 = O.welch_restated(x, sr, 1024, 512)
            _close(p2, g["psd"][u], 1e-9, 1e-300)
            _close(np.sqrt(np.mean(x ** 2)), g["rms"][u])
            _close(O.crest_factor(x), g["crest"][u])
            u += 1
    _, p = O.compute_psd_periodogram(ch[0, :4096].astype(np.float64), fs=sr, nfft=8192)
    _close(p, g["periodogram_8192"], 1e-10, 0)
    _, p = O.compute_psd_welch(ch[1, :sr].astype(np.float64), fs=sr, nperseg=2048, noverlap=1024, scaling="spectrum")
    _close(p, g["welch_2048_spectrum"], 1e-10, 0)


def test_segmentation_tables():
    g = cases.load("segmentation_tables.npz")
    n = len(g.files) // 3
    assert n == 8
    for i in range(n):
        L, sr, sec, ovl, pad, mn, nseg, seglen = g[f"a{3 * i}"]
        starts, valid = g[f"a{3 * i + 1}"], g[f"a{3 * i + 2}"]
        seg, hop, table = O.segment_table(int(L), int(sr), float(sec), float(ovl), bool(pad), None if mn < 0 else float(mn))
        assert len(table) == int(nseg)
        if table:
            assert seg == int(seglen)
        assert [t[0] for t in table] == [int(s) for s in starts]
        assert [t[1] for t in table] == [int(v) for v in valid]
