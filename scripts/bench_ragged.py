#!/usr/bin/env python
"""Ragged batches (clips of different lengths in one launch) against the two ways to do without them: the same clips padded to
the longest through the uniform entry points, and one call per clip.  Device-resident inputs, CUDA events around the device
forms, 3 warm-ups, median of 5 timed runs; every input is larger than L2.  One JSON line per measurement.

  speech   100 000 clips, lengths uniform in [8 000, 16 000] samples @ 16 kHz, MFCC13 (n_fft 512, hop 160, 40 mels)
  urban    4 000 clips of 0.2 - 4 s @ 44.1 kHz, the cfg4 feature set at 2048 / 512, one mean vector per clip (clip_vectors)
  control  the cfg3 shape (100 000 x 16 000, all lengths equal) through the ragged path and through the uniform two-kernel path
           (SYGB200_NO_RES=1); each in its own process, alternating, because the switch is read once per process
  long     8 recordings of 10 min @ 44.1 kHz as ragged units (equal lengths) against the uniform path, cfg4 features: few long
           units, the other end of the per-frame table's range

The padded path computes the padding frames too (and, for the clip vectors, aggregates over them: its vectors are wrong); it is
timed for the work it does.  The per-clip loop runs a stated subset of the clips one call each and is scaled linearly."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sygnals_b200 import _ffi, batch  # noqa: E402
from sygnals_b200.utils import synth  # noqa: E402

CFG4 = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]


def timed(fn, reps=5, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def clips_matrix(n, L, lengths, sr, seed):
    """[n, L] CUDA float32: clip u in row u, zero past lengths[u] (= the clips padded to the longest)."""
    m = torch.empty((n, L), dtype=torch.float32, device="cuda")
    synth.torch_mixture_(m, sr, seed=seed)
    ln = torch.from_numpy(lengths).cuda()
    m.masked_fill_(torch.arange(L, device="cuda")[None, :] >= ln[:, None], 0.0)
    return m


def run(name, sr, L, lengths, features, fl, hop, fp, vectors, loop_subset):
    eng = _ffi.engine(0)
    n = len(lengths)
    m = clips_matrix(n, L, lengths, sr, seed=7)
    y = m.view(-1)
    starts = np.arange(n, dtype=np.int64) * L
    p = _ffi.make_params(eng.lib, sr, features, fl, hop, feature_params=fp)
    rows = eng.rows(p)
    units = eng.ragged_units(starts, lengths, y.numel())
    F = int(eng.lib.ragged_frame_offsets(units, fl, hop)[-1])
    T = eng.frame_count(L, fl, hop)
    st = torch.cuda.current_stream().cuda_stream
    audio_s = float(lengths.sum()) / sr
    if vectors:
        ids = [0] * rows
        out_r = torch.empty((n, rows), dtype=torch.float64, device="cuda")
        rag = lambda: eng.segment_vectors_ragged_dev(y.data_ptr(), units, p, ids, out_r.data_ptr(), st)
        out_p = torch.empty((n, rows), dtype=torch.float64, device="cuda")
        pad = lambda: eng.segment_vectors_dev(y.data_ptr(), eng.units_clips(n, L), p, ids, out_p.data_ptr(), st)
    else:
        out_r = torch.empty((rows, F), dtype=torch.float32, device="cuda")
        rag = lambda: eng.features_ragged_dev(y.data_ptr(), units, p, out_r.data_ptr(), st)
        out_p = torch.empty((n, rows, T), dtype=torch.float32, device="cuda")
        pad = lambda: eng.features_dev(y.data_ptr(), eng.units_clips(n, L), p, out_p.data_ptr(), st)
    ms_r = timed(rag)
    ms_p = timed(pad)
    print(json.dumps({"workload": name, "path": "ragged", "clips": n, "frames": F, "ms": ms_r, "audio_s_per_s": audio_s / (ms_r * 1e-3)}),
          flush=True)
    print(json.dumps({"workload": name, "path": "padded uniform", "clips": n, "frames": n * T, "ms": ms_p,
                      "audio_s_per_s": audio_s / (ms_p * 1e-3), "frame_ratio": n * T / F, "time_ratio": ms_p / ms_r}), flush=True)
    # one call per clip over the first `loop_subset` clips, scaled linearly to all clips
    k = loop_subset
    one_out = torch.empty((rows, T), dtype=torch.float64 if vectors else torch.float32, device="cuda")

    def loop():
        for u in range(k):
            ptr = y.data_ptr() + 4 * int(starts[u])
            un = eng.units_clips(1, int(lengths[u]))
            if vectors:
                eng.segment_vectors_dev(ptr, un, p, [0] * rows, one_out.data_ptr(), st)
            else:
                eng.features_dev(ptr, un, p, one_out.data_ptr(), st)
    ms_l = timed(loop, reps=3, warm=1) * n / k
    print(json.dumps({"workload": name, "path": "per-clip loop", "clips": n, "subset": k, "scaling": f"linear x{n / k:g}",
                      "ms": ms_l, "audio_s_per_s": audio_s / (ms_l * 1e-3), "time_ratio": ms_l / ms_r}), flush=True)
    del m, y, out_r, out_p
    torch.cuda.empty_cache()


def control(path):
    eng = _ffi.engine(0)
    sr, n, L = 16000, 100000, 16000
    m = torch.empty((n, L), dtype=torch.float32, device="cuda")
    synth.torch_mixture_(m, sr, seed=3)
    p = _ffi.make_params(eng.lib, sr, ["mfcc"], 512, 160, feature_params={"mfcc": {"n_mels": 40}})
    rows, T = eng.rows(p), eng.frame_count(L, 512, 160)
    st = torch.cuda.current_stream().cuda_stream
    out = torch.empty((n * rows * T,), dtype=torch.float32, device="cuda")
    if path == "ragged":
        units = eng.ragged_units(np.arange(n, dtype=np.int64) * L, np.full(n, L, np.int64), n * L)
        fn = lambda: eng.features_ragged_dev(m.data_ptr(), units, p, out.data_ptr(), st)
    else:
        fn = lambda: eng.features_dev(m.data_ptr(), eng.units_clips(n, L), p, out.data_ptr(), st)
    ms = timed(fn)
    print(json.dumps({"workload": "control", "path": path, "SYGB200_NO_RES": os.environ.get("SYGB200_NO_RES", ""), "clips": n,
                      "frames": n * T, "ms": ms, "audio_s_per_s": n * 1.0 / (ms * 1e-3),
                      "resident": eng.lib.dll.syg_debug_last_features_resident()}), flush=True)


def long_units():
    eng = _ffi.engine(0)
    sr, n, L = 44100, 8, 600 * 44100
    m = torch.empty((n, L), dtype=torch.float32, device="cuda")
    synth.torch_mixture_(m, sr, seed=5)
    p = _ffi.make_params(eng.lib, sr, CFG4, 2048, 512)
    rows, T = eng.rows(p), eng.frame_count(L, 2048, 512)
    st = torch.cuda.current_stream().cuda_stream
    out = torch.empty((n * rows * T,), dtype=torch.float32, device="cuda")
    units = eng.ragged_units(np.arange(n, dtype=np.int64) * L, np.full(n, L, np.int64), n * L)
    for path, fn in (("ragged", lambda: eng.features_ragged_dev(m.data_ptr(), units, p, out.data_ptr(), st)),
                     ("uniform", lambda: eng.features_dev(m.data_ptr(), eng.units_clips(n, L), p, out.data_ptr(), st))) * 2:
        ms = timed(fn)
        print(json.dumps({"workload": "long", "path": path, "clips": n, "frames": n * T, "ms": ms, "audio_s_per_s": n * 600.0 / (ms * 1e-3)}),
              flush=True)
    del m, out
    torch.cuda.empty_cache()


def main():
    if len(sys.argv) > 2 and sys.argv[1] == "--control":
        control(sys.argv[2])
        return
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}), flush=True)
    rng = np.random.default_rng(2024)
    run("speech", 16000, 16000, rng.integers(8000, 16001, 100000).astype(np.int64), ["mfcc"], 512, 160, {"mfcc": {"n_mels": 40}},
        vectors=False, loop_subset=500)
    rng = np.random.default_rng(2025)
    run("urban", 44100, 176400, rng.integers(8820, 176401, 4000).astype(np.int64), CFG4, 2048, 512, None, vectors=True, loop_subset=200)
    long_units()
    for _ in range(3):                                       # alternating, separate processes
        for path, env in (("ragged", {}), ("uniform", {"SYGB200_NO_RES": "1"})):
            subprocess.run([sys.executable, os.path.abspath(__file__), "--control", path], env={**os.environ, **env}, check=True)


if __name__ == "__main__":
    main()
