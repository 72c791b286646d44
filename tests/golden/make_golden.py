"""
Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference, with librosa replaced
by oracle/librosa_shim.py -- librosa itself is not installable offline) on small versions of the five
BASELINE.json configs.  Run in the build container only:

    python tests/golden/make_golden.py

Inputs are regenerated from seeds by sygnals_b200/utils/synth.py; each file stores a float64 checksum of
its input so drift of the generator is detected.
"""
import logging
import os
import sys
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402
from sygnals_b200.utils import synth  # noqa: E402

warnings.simplefilter("ignore")
logging.disable(logging.CRITICAL)
ref_loader.load_reference()
from sygnals.core.dsp import compute_psd_periodogram, compute_psd_welch, compute_stft  # noqa: E402
from sygnals.core.features.manager import extract_features  # noqa: E402
from sygnals.core.features.time_domain import crest_factor  # noqa: E402
from sygnals.core.segmentation import segment_fixed_length  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
CFG4_FEATURES = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]


def checksum(x):
    x = np.asarray(x, dtype=np.float64).ravel()
    return np.array([x.sum(), np.abs(x).sum(), (x * np.arange(1, x.size + 1)).sum()])


def stack(d, skip=("time",)):
    names = [k for k in d if k not in skip]
    return names, np.stack([d[k] for k in names])


def main():
    # cfg1: 10 s @ 22.05 kHz, MFCC(128 mels, 20 coeffs) + RMS
    sr = 22050
    y = synth.mixture(10 * sr, sr, seed=101)
    r = extract_features(y.astype(np.float64), sr, ["mfcc", "rms_energy"], frame_length=2048, hop_length=512,
                         feature_params={"mfcc": {"n_mels": 128, "n_mfcc": 20}}, output_format="dict_of_arrays")
    names, rows = stack(r)
    np.savez_compressed(os.path.join(OUT, "cfg1_mfcc_rms.npz"), names=np.array(names), rows=rows, time=r["time"],
                        in_checksum=checksum(y), sr=sr, seed=101)

    # cfg2 (small): STFT sweep, 2 clips x 8000 samples @ 16 kHz
    sr = 16000
    clips = np.stack([synth.mixture(8000, sr, seed=202), synth.edge_clip("impulse", 8000, sr)])
    d = {"in_checksum": checksum(clips), "sr": sr}
    for n_fft in (256, 512, 1024, 2048, 4096, 8192):
        for c in range(clips.shape[0]):
            D = compute_stft(clips[c].astype(np.float64), n_fft=n_fft, hop_length=n_fft // 4)
            d[f"D_{n_fft}_{c}"] = D.astype(np.complex64)
    np.savez_compressed(os.path.join(OUT, "cfg2_stft_sweep.npz"), **d)
    d = {"in_checksum": checksum(clips), "sr": sr}                       # own file: each golden file stays under 1 MB
    D = compute_stft(clips[0].astype(np.float64), n_fft=1024, hop_length=200, win_length=800, pad_mode="reflect")
    d["D_reflect_1024_800_200"] = D.astype(np.complex64)
    D = compute_stft(clips[0].astype(np.float64), n_fft=512, hop_length=128, center=False)
    d["D_nocenter_512_128"] = D.astype(np.complex64)
    np.savez_compressed(os.path.join(OUT, "cfg2_stft_variants.npz"), **d)

    # cfg3 (small): speech-commands shape, 6 edge clips + 4 mixtures, 1 s @ 16 kHz
    clips = synth.clip_batch(10, 16000, 16000, seed=303, edges=True)
    rows = []
    for c in clips:
        r = extract_features(c.astype(np.float64), 16000, ["mfcc"], frame_length=512, hop_length=160,
                             feature_params={"mfcc": {"n_mels": 40}}, output_format="dict_of_arrays")
        names, m = stack(r)
        rows.append(m)
    np.savez_compressed(os.path.join(OUT, "cfg3_speech_mfcc.npz"), names=np.array(names), rows=np.stack(rows),
                        time=r["time"], in_checksum=checksum(clips), sr=16000, seed=303)

    # cfg4 (small): 7.3 s @ 44.1 kHz, 2 s segments, 50 % overlap, pad -> 8 segments, 24 feature rows
    sr = 44100
    y = synth.long_signal(int(7.3 * sr), sr, seed=404)
    segs = segment_fixed_length(y.astype(np.float64), sr, 2.0, overlap_ratio=0.5, pad=True)
    rows = []
    for s in segs:
        r = extract_features(s, sr, CFG4_FEATURES, frame_length=2048, hop_length=512, output_format="dict_of_arrays")
        names, m = stack(r)
        rows.append(m)
    np.savez_compressed(os.path.join(OUT, "cfg4_env_sound.npz"), names=np.array(names), rows=np.stack(rows),
                        time=r["time"], n_segments=len(segs), seg_len=len(segs[0]),
                        last_segment_tail=segs[-1][-4:], in_checksum=checksum(y), sr=sr, seed=404)

    # cfg5 (small): 3 channels x 2 s @ 25.6 kHz, Welch-1024 + RMS + crest per channel-second
    sr = 25600
    ch = np.stack([synth.long_signal(2 * sr, sr, seed=505 + c, block_sec=0.5) for c in range(3)])
    psd, rms, crest = [], [], []
    for c in range(ch.shape[0]):
        for w in range(2):
            x = ch[c, w * sr:(w + 1) * sr].astype(np.float64)
            f, p = compute_psd_welch(x, fs=sr, window="hann", nperseg=1024, noverlap=512, detrend="constant",
                                     scaling="density")
            psd.append(p)
            rms.append(np.sqrt(np.mean(x ** 2)))
            crest.append(crest_factor(x))
    f2, p2 = compute_psd_periodogram(ch[0, :4096].astype(np.float64), fs=sr, window="hann", nfft=8192)
    f3, p3 = compute_psd_welch(ch[1, :sr].astype(np.float64), fs=sr, window="hann", nperseg=2048, noverlap=1024,
                               scaling="spectrum")
    np.savez_compressed(os.path.join(OUT, "cfg5_machinery_psd.npz"), freqs=f, psd=np.stack(psd), rms=np.array(rms),
                        crest=np.array(crest), periodogram_8192=p2, welch_2048_spectrum=p3,
                        in_checksum=checksum(ch), sr=sr, seed=505)

    # segmentation boundary table (integer-exact)
    cases = []
    for (L, srr, sec, ovl, pad, mn) in [(5300, 1000, 1.0, 0.25, True, None), (5300, 1000, 1.0, 0.5, False, None),
                                        (5300, 1000, 0.7, 0.3, True, 0.2), (1000, 1000, 2.0, 0.0, True, None),
                                        (1000, 1000, 2.0, 0.0, False, None), (88200 * 3 + 17, 44100, 2.0, 0.5, True, None),
                                        (4096, 22050, 0.01, 0.9, True, None), (10, 1000, 0.001, 0.0, True, None)]:
        y = np.arange(1, L + 1, dtype=np.float64)
        segs = segment_fixed_length(y, srr, sec, overlap_ratio=ovl, pad=pad, min_segment_length_sec=mn)
        starts = [int(s[0]) - 1 for s in segs]
        valid = [int(np.count_nonzero(s)) for s in segs]
        seglen = len(segs[0]) if segs else 0
        cases.append(np.array([L, srr, sec, ovl, int(pad), -1 if mn is None else mn, len(segs), seglen], dtype=np.float64))
        cases.append(np.array(starts, dtype=np.float64))
        cases.append(np.array(valid, dtype=np.float64))
    np.savez_compressed(os.path.join(OUT, "segmentation_tables.npz"), **{f"a{i}": c for i, c in enumerate(cases)})
    for fn in sorted(os.listdir(OUT)):
        if fn.endswith(".npz"):
            print(fn, os.path.getsize(os.path.join(OUT, fn)))


if __name__ == "__main__":
    main()
