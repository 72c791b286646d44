#!/usr/bin/env python
"""Per-channel Welch PSDs of a multi-channel PCM recording, end to end from pinned host memory (BASELINE cfg5 shape: 64 channels x
600 s at 25.6 kHz, one 1 s window per (channel, second), nperseg 1024, noverlap 512, hann, density, RMS / crest / peak).

Three arms, alternated in one process, wall clock around calls that return their results in host memory, 1 warm-up each, median
of --reps runs:
  a  syg_psd_welch_host_pcm_channels on the interleaved s16 payload (2 bytes per sample cross PCIe, planar ingest on the device)
  b  syg_psd_welch_host_f32 on the channel-major float32 buffer (4 bytes per sample): the path bench.py's cfg5 e2e arm times
  c  as a, with an s24 payload (3 bytes per sample)
The s16 payload is the float signal quantised; (b)'s input is exactly s16 / 32768 and (c)'s codes are the s16 codes times 256, so
all three arms compute from the same float32 samples and must agree bit for bit.  The payloads (1.97 GB s16) are larger than L2.

Also timed: the planar ingest kernel alone on the device-resident payload (CUDA events, median of --reps launches), against the
HBM bound (BPS + 4) bytes per sample / 7.7 TB/s.  Card name and power limit are read in the same run.  Prints one JSON line; --out
also writes it to a file."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sygnals_b200 import _ffi  # noqa: E402
from sygnals_b200.utils import synth  # noqa: E402

HBM_BPS = 7.7e12          # HGX B200 data sheet, one GPU


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name(0)


def pinned(t):
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--seconds", type=int, default=600)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    sr, C, S = 25600, args.channels, args.seconds
    T = S * sr
    eng = _ffi.engine(0)
    dev = torch.device("cuda", 0)

    y = torch.empty((C * S, sr), dtype=torch.float32, device=dev)           # channel c, second s in row c * S + s
    synth.torch_mixture_(y, sr, seed=31)
    q = torch.clamp(torch.round(y.view(C, T) * 32768.0), -32768, 32767).to(torch.int16)
    del y
    f32 = pinned(q.float() / 32768.0)                                       # [C, T] channel-major float32 (arm b's input)
    inter = q.t().contiguous()                                              # [T, C] interleaved frames
    s16 = pinned(inter.view(torch.uint8).view(-1))
    s24 = pinned((inter.to(torch.int32) * 256).view(torch.uint8).view(T, C, 4)[:, :, :3].contiguous().view(-1))
    del inter
    torch.cuda.synchronize()

    wins = eng.units_clips(S, sr)                                           # windows over the frames, shared by all channels
    units_f32 = eng.units_clips(C * S, sr)
    wel = (float(sr), 0, 1024, 512, 1024, True, 0)
    f32_np = f32.numpy().reshape(-1)
    arms = {
        "a_s16_channels": lambda: eng.psd_welch_host_pcm_channels(s16.data_ptr(), _ffi.PCM_S16, C, wins, *wel, stats=True),
        "b_f32_channel_major": lambda: eng.psd_welch_host(f32_np, units_f32, *wel, stats=True),
        "c_s24_channels": lambda: eng.psd_welch_host_pcm_channels(s24.data_ptr(), _ffi.PCM_S24, C, wins, *wel, stats=True),
    }
    h2d = {"a_s16_channels": C * T * 2, "b_f32_channel_major": C * T * 4, "c_s24_channels": C * T * 3}
    out = {k: fn() for k, fn in arms.items()}                               # warm-up, and the results compared below
    pa, sa = out["a_s16_channels"]
    pb, sb = out["b_f32_channel_major"]
    pc, sc = out["c_s24_channels"]
    pb = pb.reshape(C, S, -1).transpose(1, 0, 2)                            # channel-major units -> [window][channel]
    sb = sb.reshape(C, S, 3).transpose(1, 0, 2)
    same_ab = bool(np.array_equal(pa, pb) and np.array_equal(sa, sb) and pa.tobytes() == np.ascontiguousarray(pb).tobytes())
    same_ac = bool(pa.tobytes() == pc.tobytes() and sa.tobytes() == sc.tobytes())

    times = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            times[k].append(time.perf_counter() - t0)
    res = {}
    for k in arms:
        dt = float(np.median(times[k]))
        res[k] = {"ms": 1e3 * dt, "channel_s_per_s": C * S / dt, "h2d_bytes": h2d[k], "h2d_gbs": h2d[k] / dt / 1e9,
                  "runs_ms": [round(1e3 * t, 2) for t in times[k]]}

    kern = {}
    for name, fmt, host in (("s16", _ffi.PCM_S16, s16), ("s24", _ffi.PCM_S24, s24)):
        d_raw = host.to(dev)
        d_out = torch.empty(C * _ffi.plane_pitch(T), dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream().cuda_stream
        eng.ingest_pcm_channels_dev(d_raw.data_ptr(), fmt, C, T, d_out.data_ptr(), stream)
        ts = []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eng.ingest_pcm_channels_dev(d_raw.data_ptr(), fmt, C, T, d_out.data_ptr(), stream)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ms = float(np.median(ts))
        bps = _ffi.PCM_BYTES[fmt]
        bound_ms = (bps + 4) * C * T / HBM_BPS * 1e3
        planes = d_out.view(C, -1)[:, :T]
        exact = bool(torch.equal(planes, f32.to(dev)))
        kern[name] = {"ms": ms, "hbm_bytes": (bps + 4) * C * T, "gbs": (bps + 4) * C * T / (ms * 1e-3) / 1e9,
                      "hbm_bound_ms": bound_ms, "share_of_hbm_bound": bound_ms / ms, "planes_equal_f32_input": exact}
        del d_raw, d_out

    line = {"metric": "channel-sec/sec (cfg5 Welch PSD + RMS/crest, host payload to host result)", "unit": "channel-s/s",
            "card": card(), "config": {"channels": C, "seconds": S, "sr": sr, "nperseg": 1024, "noverlap": 512, "nfft": 1024,
                                       "reps": args.reps, "timing": "wall clock around each host call, median, arms alternated"},
            "arms": res, "a_equals_b_bit_for_bit": same_ab, "a_equals_c_bit_for_bit": same_ac,
            "speedup_a_over_b": res["b_f32_channel_major"]["ms"] / res["a_s16_channels"]["ms"], "planar_ingest_kernel": kern}
    s = json.dumps(line)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")
    if not (same_ab and same_ac):
        sys.exit("the arms disagree")


if __name__ == "__main__":
    main()
