#!/usr/bin/env python
"""Log-mel spectrograms (syg_mel_spectrogram_f32, db = 1) of two dataset-image shapes, inputs resident in HBM:
  cfg3  100 000 clips of 1 s at 16 kHz, n_fft 512, hop 160, 40 mels            (speech commands)
  cfg4  36 000 segments of 2 s at 44.1 kHz, 50 % overlap, n_fft 2048, hop 512, 128 mels   (segments of a 10 h recording)

Per shape, CUDA events around each call, --warmup calls first, median of --reps:
  mel           the call: frame kernel (mel energies + unit maxima to the workspace) + mel_store_kernel (dB, transpose, store)
  kernels       the engine's per-launch timing (syg_ctx_profile_*) in a separate pass: frame kernel and mel_store_kernel alone;
                mel_store's bytes are the workspace read plus the output write, 8 bytes per output float
  mfcc          the existing MFCC-only feature call (13 coefficients) on the same inputs
  torchaudio    MelSpectrogram + AmplitudeToDB(top_db=80) in batches of units: a yardstick, not the reference (its dB is
                relative to 1.0 with the clamp over the batch, and it materialises the complex STFT)
Algorithmic bytes = 4 x unique input samples + 4 x output floats; the HBM bound is those bytes over 7.7 TB/s (HGX B200 data sheet,
one GPU).  Unit 0 of each shape is checked against the float64 oracle's mel stage.  Card name and power limit are read in the
same run.  Prints one JSON line; --out also writes it to a file."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import sygnals_oracle as orc  # noqa: E402
from sygnals_b200 import _ffi, batch  # noqa: E402
from sygnals_b200.utils import synth  # noqa: E402

HBM_BPS = 7.7e12          # HGX B200 data sheet, one GPU


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name(0)


def oracle_log_mel(y, sr, fl, hop, n_mels):
    """float64 power_to_db(S_mel, ref=np.max) of y with the oracle's librosa, as extract_features builds it (manager.py:184-223)"""
    L = orc.librosa
    S = np.abs(L.stft(y=y, n_fft=fl, hop_length=hop, win_length=fl, window="hann", center=True)).astype(np.float64)
    return L.power_to_db(L.feature.melspectrogram(S=S ** 2.0, sr=sr, n_mels=n_mels, fmin=0.0, fmax=sr / 2.0, n_fft=fl), ref=np.max)


def timed(fn, warmup, reps):
    """median ms of fn() between CUDA events on the current stream"""
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), [round(t, 3) for t in ts]


def shape(name, eng, args):
    if name == "cfg3":
        sr, fl, hop, n_mels = 16000, 512, 160, 40
        n, L = args.cfg3_clips, sr
        y = torch.empty((n, L), dtype=torch.float32, device="cuda")
        synth.torch_mixture_(y, sr, seed=303)
        units = eng.units_clips(n, L)
        unique = n * L
        audio_s = n * L / sr
        unit = lambda u: y[u]                                                   # noqa: E731
        windows = lambda u0, u1: y[u0:u1]                                       # noqa: E731
    else:
        sr, fl, hop, n_mels = 44100, 2048, 512, 128
        seg_len, seg_hop, n = 2 * sr, sr, args.cfg4_segments
        total = (n - 1) * seg_hop + seg_len
        y = torch.empty(total, dtype=torch.float32, device="cuda")
        synth.torch_recording_(y, 0, sr, seed=404)
        units = eng.units_clips(n, seg_len, total_len=total, stride=seg_hop)
        L, unique = seg_len, total
        audio_s = n * seg_len / sr
        unit = lambda u: y[u * seg_hop:u * seg_hop + seg_len]                   # noqa: E731
        windows = lambda u0, u1: y[u0 * seg_hop:(u1 - 1) * seg_hop + seg_len].unfold(0, seg_len, seg_hop)   # noqa: E731
    torch.cuda.synchronize()
    T = eng.frame_count(L, fl, hop)
    stream = torch.cuda.current_stream().cuda_stream
    p = batch._mel_params(eng.lib, sr, fl, hop, True, "hann", n_mels, 0.0, None, 2.0)
    out = torch.empty((n, n_mels, T), dtype=torch.float32, device="cuda")
    call = lambda: eng.mel_spectrogram_dev(y.data_ptr(), units, p, True, out.data_ptr(), stream)   # noqa: E731
    ms, runs = timed(call, args.warmup, args.reps)
    resident = eng.lib.dll.syg_debug_last_features_resident()
    fk = eng.lib.dll.syg_debug_last_feature_kernel()

    eng.profile_enable(True)
    eng.profile_read(reset=True)
    for _ in range(args.reps):
        call()
    torch.cuda.synchronize()
    prof = eng.profile_read(reset=True)
    eng.profile_enable(False)
    frame_ms = prof["frame"][0] / args.reps
    store_ms = prof["finalize"][0] / args.reps

    ref = oracle_log_mel(unit(0).cpu().numpy().astype(np.float64), sr, fl, hop, n_mels)
    err0 = float(np.abs(out[0].cpu().numpy() - ref).max())

    pm = _ffi.make_params(eng.lib, sr, ["mfcc"], fl, hop, feature_params={"mfcc": {"n_mels": n_mels}})
    mf = torch.empty((n, 13, T), dtype=torch.float32, device="cuda")
    mfcc_ms, mfcc_runs = timed(lambda: eng.features_dev(y.data_ptr(), units, pm, mf.data_ptr(), stream), args.warmup, args.reps)
    mfcc_resident = eng.lib.dll.syg_debug_last_features_resident()
    del mf

    import torchaudio
    ta = torch.nn.Sequential(
        torchaudio.transforms.MelSpectrogram(sample_rate=sr, n_fft=fl, hop_length=hop, n_mels=n_mels, power=2.0, center=True,
                                             pad_mode="constant", norm="slaney", mel_scale="slaney"),
        torchaudio.transforms.AmplitudeToDB(stype="power", top_db=80.0)).cuda()
    step = max(1, int(args.ta_stft_gb * 2**30 // ((fl // 2 + 1) * T * 8)))     # units per batch: the complex STFT within --ta-stft-gb

    def ta_all():
        with torch.no_grad():
            for u0 in range(0, n, step):
                ta(windows(u0, min(n, u0 + step)))
    ta_ms, ta_runs = timed(ta_all, 1, max(1, args.reps // 2))

    out_floats = n * n_mels * T
    alg_bytes = 4 * unique + 4 * out_floats
    store_bytes = 8 * out_floats
    res = {
        "units": n, "unit_len": L, "sr": sr, "n_fft": fl, "hop": hop, "n_mels": n_mels, "T": T, "audio_s": audio_s,
        "output_bytes": 4 * out_floats, "feature_kernel": fk, "resident": resident,
        "mel": {"ms": ms, "audio_s_per_s": audio_s / (ms * 1e-3), "runs_ms": runs,
                "algorithmic_bytes": alg_bytes, "hbm_bound_ms": alg_bytes / HBM_BPS * 1e3,
                "share_of_hbm_bound": alg_bytes / HBM_BPS / (ms * 1e-3)},
        "kernels": {"frame_ms": frame_ms, "mel_store_ms": store_ms, "mel_store_bytes": store_bytes,
                    "mel_store_gbs": store_bytes / (store_ms * 1e-3) / 1e9,
                    "mel_store_share_of_hbm": store_bytes / HBM_BPS / (store_ms * 1e-3)},
        "mfcc_only": {"ms": mfcc_ms, "audio_s_per_s": audio_s / (mfcc_ms * 1e-3), "resident": mfcc_resident, "runs_ms": mfcc_runs},
        "torchaudio_yardstick": {"ms": ta_ms, "audio_s_per_s": audio_s / (ta_ms * 1e-3), "units_per_batch": step, "runs_ms": ta_runs,
                                 "note": "yardstick, not the reference: dB relative to 1.0, clamp over the batch"},
        "unit0_max_abs_db_error_vs_oracle": err0,
    }
    del y, out
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="cfg3,cfg4")
    ap.add_argument("--cfg3-clips", type=int, default=100_000)
    ap.add_argument("--cfg4-segments", type=int, default=36_000)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--ta-stft-gb", type=float, default=4.0, help="torchaudio arm: complex STFT bytes per batch of units")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    eng = _ffi.engine(0)
    line = {"metric": "log-mel spectrogram, audio-sec/sec (inputs and outputs in HBM)", "unit": "audio-s/s", "card": card(),
            "config": {"timing": "CUDA events around each call, median", "warmup": args.warmup, "reps": args.reps},
            "shapes": {s: shape(s, eng, args) for s in args.shapes.split(",")}}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
