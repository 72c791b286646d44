#!/usr/bin/env python
"""bench.py -- throughput of the Sygnals segment->features hot path on B200 (see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg4|cfg1|cfg2|cfg3|cfg5] [--impl native|reference]
                    [--dump-outputs DIR]

Default workload = BASELINE.json configs[3] ("cfg4", the config the metric "audio-sec/sec (MFCC+spectral feats)" names):
ONE 10 h synthetic 44.1 kHz recording, fixed-length 2 s segments with 50 % overlap (36 000 segments), per segment
MFCC(13) + spectral contrast(7) + centroid + rolloff + RMS + crest over 2048/512 frames, then the `sygnals save dataset`
assembly (format_feature_vectors_per_segment, mean over the segment's frames) -> float64 [36000, 24].

One "step" = one pass of the product path over the recording resident in HBM: `dist.run_shard` (fused frame kernels + on-device
aggregation) on this rank's block of segments (its sample range + a 44 100-sample halo) followed by `dist.gather_features` (one
NCCL all-gather of the [segments, 24] vectors) -- STRONG scaling: the 10 h are split over the N ranks, the collective is inside
the timed region.  `value` = 36 000 audio-seconds x steps / max-over-ranks device time.  A weak-scaling figure (10 h per rank, no
collective: round 1's measure) is reported under `weak`.

`e2e` = the same path through the C ABI with HOST buffers: the recording as 16-bit PCM in pinned memory (what a WAV file holds)
-> H2D -> ingest + kernels + aggregation -> D2H of the vectors, wall clock, max over ranks.

`--impl reference` times the reference's CPU algorithm (oracle/: the reference's own call graph restated on numpy/scipy,
float64, incl. its per-frame Python loops; librosa itself is not installable offline) on the host cores.

Other workloads (secondary lines, same contract): cfg3 speech-commands MFCC, cfg2 STFT magnitude sweep, cfg5 Welch PSD.

`--dump-outputs DIR` writes what the timed path computed in its last timed step as DIR/<name>.npy (see `dump_outputs`).  The
inputs are synthesised from fixed seeds, so two builds run with the same arguments can be compared output for output.  cfg4 and
cfg1/cfg3 write the output gathered from all ranks; cfg2 and cfg5 have no collective, so under --gpus N > 1 they write rank 0's
block (its clips / channels, whose inputs are seeded per rank).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CFG4_FEATURES = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]
CFG2_NFFT = [256, 512, 1024, 2048, 4096, 8192]

WORKLOADS = {
    "cfg4": dict(kind="segments", metric="audio-sec/sec (MFCC+spectral feats)", unit="audio-s/s",
                 desc="env-sound: ONE 10 h @ 44.1 kHz recording, 2 s segments, 50% overlap, MFCC13+contrast7+centroid+rolloff+rms+crest, "
                      "n_fft 2048 hop 512, mean over each segment's frames",
                 sr=44100, seg_sec=2.0, overlap=0.5, hours=10.0, features=CFG4_FEATURES, fl=2048, hop=512, fp=None),
    "cfg1": dict(kind="clips", metric="audio-sec/sec (MFCC+RMS, one clip per call)", unit="audio-s/s",
                 desc="the reference's CPU case: ONE 10 s @ 22.05 kHz clip per call, MFCC20 (n_fft 2048, hop 512, 128 mels) + RMS",
                 sr=22050, clip=220500, n_clips=1, features=["mfcc", "rms_energy"], fl=2048, hop=512,
                 fp={"mfcc": {"n_mels": 128, "n_mfcc": 20}}),
    "cfg3": dict(kind="clips", metric="audio-sec/sec (MFCC)", unit="audio-s/s",
                 desc="speech-commands: 100k x 1 s @ 16 kHz clips, MFCC13, n_fft 512 hop 160, 40 mels",
                 sr=16000, clip=16000, n_clips=100000, features=["mfcc"], fl=512, hop=160, fp={"mfcc": {"n_mels": 40}}),
    "cfg2": dict(kind="stft", metric="audio-sec/sec (STFT magnitude)", unit="audio-s/s",
                 desc="STFT magnitude sweep n_fft 256..8192 (hop n_fft/4, hann, centred), 4096 x 1 s @ 16 kHz clips",
                 sr=16000, clip=16000, n_clips=4096),
    "cfg5": dict(kind="welch", metric="channel-sec/sec (Welch PSD + RMS/crest)", unit="channel-s/s",
                 desc="machinery: 64 channels @ 25.6 kHz, per 1 s window Welch PSD (nperseg 1024, noverlap 512, hann, density) + RMS + crest",
                 sr=25600, channels=64, seconds=600),
}

_REAL_STDOUT = None


def guard_stdout():
    """stdout carries exactly ONE JSON line.  Native libraries write banners straight to file descriptor 1 (NCCL prints its version
    there whenever NCCL_DEBUG is set), so fd 1 is pointed at stderr for the whole run and the JSON goes out through a saved copy."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_json(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


DUMP_BYTES = 60 << 20                                                  # under 64 MB with the .npy headers
DUMP_SEED = 20240607


def dump_outputs(out_dir, arrays: dict, budget: int = DUMP_BYTES) -> None:
    """Writes each tensor of ``arrays`` (float32 / float64, leading axis = units: segments, clips, channel-seconds) to
    ``out_dir/<name>.npy``.  When they hold more than ``budget`` bytes in all, each keeps the same fraction of its units, a fixed
    seeded sample in ascending order, so that the files of two runs with the same arguments hold the same units."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = sum(t.numel() * t.element_size() for t in arrays.values())
    for name, t in arrays.items():
        n = t.shape[0]
        if total > budget:
            k = max(1, n * budget // total)
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, k, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        a = t.detach().cpu().numpy()
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {name} is {a.dtype}, expected float32 or float64")
        np.save(os.path.join(out_dir, name + ".npy"), a)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _cpu_worker(args):
    """One oracle call on one unit (runs in a pool worker)."""
    kind, x, w = args
    from oracle import sygnals_oracle as orc
    import numpy as np
    x = x.astype(np.float64)
    if kind in ("segments", "clips"):
        r = orc.extract_features(x, w["sr"], list(w["features"]), frame_length=w["fl"], hop_length=w["hop"], feature_params=w["fp"])
        if kind == "segments":                                         # + the dataset assembly of the product path
            d = {k: v for k, v in r.items() if k != "time"}
            T = len(next(iter(d.values())))
            return float(np.nansum(orc.format_feature_vectors_per_segment(d, [(0, T)], "mean")))
        return sum(float(v.sum()) for k, v in r.items() if k != "time" and v.size)
    if kind == "stft":
        return sum(float(np.abs(orc.compute_stft(x, n_fft=n, hop_length=n // 4)).sum()) for n in CFG2_NFFT)
    f, pxx = orc.compute_psd_welch(x, fs=w["sr"], window="hann", nperseg=1024, noverlap=512)
    return float(pxx.sum()) + float(np.sqrt(np.mean(x * x))) + float(orc.crest_factor(x))


def cpu_reference_run(workload: str, n_units: int, steps: int, warmup: int, procs: int | None = None):
    """Times the oracle (CPU restatement of the reference path) on `n_units` units per step with a process pool over
    all usable host cores.  Returns (seconds per step list, cores, unit description)."""
    import multiprocessing as mp
    import numpy as np
    from oracle import sygnals_oracle as orc
    from sygnals_b200.utils import synth
    w = WORKLOADS[workload]
    sr, kind = w["sr"], w["kind"]
    cores = procs or len(os.sched_getaffinity(0))
    if kind == "segments":
        seg_len = int(w["seg_sec"] * sr)
        seg_hop = max(1, int(seg_len * (1.0 - w["overlap"])))
        y = synth.long_signal(seg_hop * (n_units - 1) + seg_len, sr, seed=4321)
        units = orc.segment_fixed_length(y.astype(np.float64), sr, w["seg_sec"], overlap_ratio=w["overlap"], pad=False)[:n_units]
        what = f"{n_units} x {w['seg_sec']} s segments per step through oracle.extract_features + format_feature_vectors_per_segment"
    elif kind in ("clips", "stft"):
        units = list(synth.clip_batch(n_units, w["clip"], sr, seed=99, edges=False))
        what = f"{n_units} x {w['clip'] / sr:g} s clips per step through oracle." + ("extract_features" if kind == "clips" else "compute_stft (6 sizes)")
    else:
        units = [synth.long_signal(sr, sr, seed=700 + i, block_sec=0.25) for i in range(n_units)]
        what = f"{n_units} channel-seconds per step through oracle.compute_psd_welch + rms + crest_factor"
    assert len(units) == n_units, (len(units), n_units)
    wl = {k: v for k, v in w.items() if k in ("sr", "features", "fl", "hop", "fp")}
    jobs = [(kind, np.asarray(u, dtype=np.float32), wl) for u in units]
    times = []
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, jobs[:cores], chunksize=1)                # import + plan warm-up in every worker
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            pool.map(_cpu_worker, jobs, chunksize=max(1, len(jobs) // (cores * 4)))
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
    return times, cores, what + f" (reference call graph on numpy/scipy, float64), fork pool over {cores} cores"


def unit_seconds(w) -> float:
    """unique audio (channel) seconds one unit stands for"""
    if w["kind"] == "segments":
        return w["seg_sec"] * (1.0 - w["overlap"])
    return w["clip"] / float(w["sr"]) if "clip" in w else 1.0


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    # one process per core, one thread per process: numpy/scipy/BLAS thread pools inside 16 forked workers oversubscribe the
    # host and slow the reference down ~8x (measured); the baseline should be as fast as the reference can go
    for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[v] = "1"
    w = WORKLOADS[args.workload]
    cores = len(os.sched_getaffinity(0))
    per_core = {"segments": 24, "clips": 96, "stft": 24, "welch": 256}[w["kind"]]
    n_units = args.cpu_units or max(cores * per_core, 4 * per_core)
    times, cores, what = cpu_reference_run(args.workload, n_units, args.steps, args.warmup)
    total_t = sum(times)
    mult = len(CFG2_NFFT) if w["kind"] == "stft" else 1                 # the sweep transforms every clip six times
    value = n_units * unit_seconds(w) * mult * len(times) / total_t
    line = {
        "impl": "reference", "metric": w["metric"], "value": value, "unit": w["unit"],
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {w['desc']}", "sample": f"{n_units} units per step"},
        "cpu_baseline": {"value": value, "unit": w["unit"], "cores": cores, "kind": "port", "sample": what},
        "e2e": {"value": value, "unit": w["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit_json(line)
    return 0


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi polled every 50 ms from before the warm-up to after the timed region; `stop(t0, t1)` keeps the samples whose
    timestamps fall inside the timed window [t0, t1] (wall clock) and, when the window is shorter than the polling interval (strong
    scaling at 8 GPUs: 10 steps take 44 ms), the samples taken under the same load since the warm-up began."""
    Q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index = index
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                       "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
            self.t_start = time.time()
            self.lines = []
            import threading
            self.th = threading.Thread(target=lambda: [self.lines.append(ln) for ln in self.p.stdout], daemon=True)
            self.th.start()
        except Exception:
            self.p = None

    def count(self) -> int:
        return len(self.lines) if self.p else 1 << 30

    def stop(self, t0=None, t1=None):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.th.join(timeout=2)
        import datetime
        rows = []
        for ln in list(self.lines):
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), float(f[3]), [v.lower().startswith("active") for v in f[4:8]]))
            except ValueError:
                continue
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        window = [r for r in rows if t0 is not None and t0 - 0.03 <= r[0] <= t1 + 0.03]
        scope = "timed region"
        if len(window) < 2:                                            # shorter than the polling interval: same load since the warm-up
            window = [r for r in rows if t0 is None or r[0] <= (t1 or r[0]) + 0.03]
            scope = "warm-up + timed region (the timed region is shorter than the 50 ms polling interval)"
        reasons = set()
        for r in window:
            for name, on in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4]):
                if on:
                    reasons.add(name)
        sm_sorted = sorted(r[1] for r in window)
        load = sm_sorted[len(sm_sorted) // 2:]                         # upper half: the sampler also sees idle edges
        return {"sm_mhz": load[len(load) // 2], "sm_max_mhz": max(r[2] for r in window), "reasons": sorted(reasons),
                "samples": len(window), "power_w_max": max(r[3] for r in window), "scope": scope}


# ------------------------------------------------------------------------------------------------ native arm
class Ctx:
    """rank / device / engine / timing helpers shared by the workloads"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from sygnals_b200 import _ffi
        self.torch, self.dist, self.args = torch, dist, args
        self.rank, self.world, self.local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the native arm has no CPU fallback (use --impl reference for the CPU baseline)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        from sygnals_b200.utils import numa
        self.full_affinity = os.sched_getaffinity(0)
        self.placement = None if os.environ.get("SYGB200_NO_NUMA_BIND") else numa.bind_to_device_node(self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.eng = _ffi.engine(self.local)
        if args.ws_mb:
            self.eng.set_workspace_limit(args.ws_mb << 20)
        self.warm = max(args.warmup, 3)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, v: float) -> float:
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def time_device(self, step, steps, warm=None, sample_clocks=True):
        """W untimed steps, then `steps` steps between CUDA events on the current stream, barrier + synchronize on both sides.
        Returns (max-over-ranks ms for all steps, this rank's ms, clocks, profile dict)."""
        torch = self.torch
        clocks = ClockSampler(self.local) if sample_clocks else None
        if clocks:
            clocks.start()                                             # polling runs through warm-up and timed region
        for _ in range(self.warm if warm is None else warm):
            step()
        if clocks:
            # short steps (strong scaling at 8 GPUs: 4.4 ms): keep the same load up, untimed, until the poller has delivered its
            # first samples, so that the clock record covers the load the timed steps run under (bounded: 2 s); the number of
            # extra steps is agreed across ranks (collectives inside `step` must match)
            t_w = time.time()
            while True:
                more = 1.0 if (clocks.count() < 3 and time.time() - t_w < 2.0) else 0.0
                if self.max_over_ranks(more) == 0.0:
                    break
                step()
        torch.cuda.synchronize()
        self.eng.profile_read(reset=True)
        self.eng.profile_enable(True)
        self.barrier()
        t0w = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        self.barrier()
        t1w = time.time()
        clk = clocks.stop(t0w, t1w) if clocks else None
        ms = e0.elapsed_time(e1)
        prof = self.eng.profile_read(reset=True)
        self.eng.profile_enable(False)
        return self.max_over_ranks(ms), ms, clk, prof

    def dump(self, arrays: dict) -> None:
        """--dump-outputs: rank 0 writes the outputs of the last timed step, before any later measurement reuses the device.  The
        callers pass the gathered output where the step gathers one (cfg4, cfg1/cfg3) and rank 0's own block otherwise (cfg2, cfg5)."""
        if self.args.dump_outputs and self.rank == 0:
            dump_outputs(self.args.dump_outputs, arrays)

    def time_wall(self, step, steps, warm=1):
        for _ in range(warm):
            step()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        self.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return self.max_over_ranks(dt)

    def peaks(self):
        p = {}
        try:
            p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        if "hbm_gbs" in p:
            return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        return 6650.0, "fallback (B200_PROFILING.md)"

    def traffic(self, workload):
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            if tr.get("workload") == workload:
                return {"dram_bytes_per_launch": tr["dram_bytes_read"] + tr["dram_bytes_write"],
                        "algorithmic_bytes_of_that_launch": tr["algorithmic_bytes"], "source": tr["source"]}
        except Exception:
            pass
        return None

    def cpu_baseline(self, workload):
        os.sched_setaffinity(0, self.full_affinity)                   # the CPU baseline uses every host core again
        cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload, "--steps", "1", "--warmup", "0"]
        try:
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
            return json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
        except Exception as exc:  # noqa: BLE001
            return {"value": None, "unit": WORKLOADS[workload]["unit"], "cores": None, "kind": "port", "sample": f"failed: {exc}"}

    def finish(self, line):
        if self.rank == 0:
            if self.world == 1 and not self.args.no_cpu:
                line["cpu_baseline"] = self.cpu_baseline(self.args.workload)
            emit_json(line)
        if self.world > 1:
            self.dist.destroy_process_group()
        return 0


def roofline_block(c: Ctx, alg_bytes_per_step, prof, steps, ms_rank, kernel, traffic=None, extra=None):
    peak, src = c.peaks()
    f_ms, f_n = prof["frame"] if kernel != "welch" else prof["welch"]
    achieved = alg_bytes_per_step * steps / (f_ms * 1e-3) / 1e9 if f_ms > 0 else None
    lps = f_n / steps if steps else 0
    r = {"bound": "hbm", "kernel": kernel, "achieved": achieved, "peak": peak, "unit": "GB/s",
         "frac": (achieved / peak) if achieved else None, "peak_source": src, "traffic": traffic,
         "kernel_launches_per_step": lps, "kernel_ms_per_launch": (f_ms / f_n) if f_n else None,
         "algorithmic_bytes_per_launch": (alg_bytes_per_step / lps) if lps else None,
         "kernel_ms_per_step": f_ms / steps, "kernel_share_of_step": f_ms / ms_rank if ms_rank > 0 else None,
         "algorithmic_bytes_per_step": alg_bytes_per_step, "scope": "rank 0's share of the step (one rank's launches against one GPU's peak)"}
    if extra:
        r.update(extra)
    return r


def run_segments(c: Ctx):
    """cfg4: the product's sharded path, strong scaling, gather inside the timed region."""
    import numpy as np
    from sygnals_b200 import _ffi, dist as sdist
    from sygnals_b200.utils import synth
    torch, args, eng = c.torch, c.args, c.eng
    w = WORKLOADS["cfg4"]
    sr, fl, hop = w["sr"], w["fl"], w["hop"]
    hours = args.hours if args.hours else w["hours"]
    total = int(round(hours * 3600 * sr))
    plan = sdist.plan_segments(total, sr, w["seg_sec"], w["overlap"], True, None, c.rank, c.world, eng.lib)
    n_local = plan.n_local
    n_have = plan.sample_end - plan.sample_begin
    p = _ffi.make_params(eng.lib, sr, w["features"], fl, hop, feature_params=w["fp"])
    rows, T = eng.rows(p), eng.frame_count(plan.seg_len, fl, hop, True)
    # this rank's slice of THE recording (position-addressable synthesis: every rank's slice equals that slice of the whole)
    y = torch.empty(n_have, dtype=torch.float32, device=c.dev)
    synth.torch_recording_(y, plan.sample_begin, sr, seed=1234)
    local = torch.empty((n_local, rows), dtype=torch.float64, device=c.dev)
    state = {}

    def step():
        sdist.run_shard(y, plan, sr, w["features"], fl, hop, feature_params=w["fp"], engine=eng, aggregation="mean", out=local)
        state["full"] = sdist.gather_features(local, plan)             # world 1: returns `local`

    ms_max, ms, clk, prof = c.time_device(step, args.steps)
    full = state["full"]
    c.dump({"features": full})                                          # float64 [segments, 24]
    audio_total = plan.n_units * unit_seconds(w)                        # unique audio seconds of the whole recording
    value = audio_total * args.steps / (ms_max * 1e-3)
    checksum = float(torch.nan_to_num(full).sum().item())
    gather_ms = None
    if c.world > 1:                                                     # the collective alone, for the record (it is inside ms_per_step)
        c.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            sdist.gather_features(local, plan)
        g1.record()
        torch.cuda.synchronize()
        gather_ms = c.max_over_ranks(g0.elapsed_time(g1) / 5)

    # ---- weak scaling (round 1's measure): every rank its own 10 h, frame features to the caller's buffer, no collective
    weak = None
    if not args.no_weak:
        units_w = eng.units_clips(plan.n_units, plan.seg_len, total_len=total, stride=plan.seg_hop)
        if c.world > 1:
            yw = torch.empty(total, dtype=torch.float32, device=c.dev)
            synth.torch_recording_(yw, 0, sr, seed=1234 + 17 * c.rank)
        else:
            yw = y
        outw = torch.empty((plan.n_units, rows, T), dtype=torch.float32, device=c.dev)
        stream = torch.cuda.current_stream().cuda_stream
        ws = max(1, min(args.steps, 5))
        wm_max, wm, _, wprof = c.time_device(lambda: eng.features_dev(yw.data_ptr(), units_w, p, outw.data_ptr(), stream), ws,
                                             warm=3, sample_clocks=False)
        weak = {"value": c.world * audio_total * ws / (wm_max * 1e-3), "unit": w["unit"], "ms_per_step": wm_max / ws, "steps": ws,
                "what": "10 h per rank, frame features [36000, 24, 173] float32 to the caller's buffer, no collective",
                "frame_kernel_ms_per_step": wprof["frame"][0] / ws, "finalize_ms_per_step": wprof["finalize"][0] / ws}
        del outw, yw

    # ---- end to end through the C ABI with HOST buffers: PCM16 in pinned memory -> vectors in pinned memory
    e2e = None
    if not args.no_e2e:
        units_l = eng.units_clips(n_local, plan.seg_len, total_len=n_have, stride=plan.seg_hop)
        ids = [_ffi.AGG_IDS["mean"]] * rows
        y16 = torch.empty(n_have, dtype=torch.int16, pin_memory=True)   # allocated once, reused by every step
        y16.copy_((y * 32767.0).round().clamp(-32768, 32767).to(torch.int16))
        vh = torch.empty((n_local, rows), dtype=torch.float64, pin_memory=True)
        vh_np = vh.numpy()
        gl = torch.empty((n_local, rows), dtype=torch.float64, device=c.dev)
        ne = max(1, min(args.steps, args.e2e_steps))

        def e2e_step():
            eng.segment_vectors_host(y16.data_ptr(), units_l, p, ids, out=vh_np, fmt=_ffi.PCM_S16, channels=1)
            if c.world > 1:                                             # dataset assembly across ranks: vectors back to HBM, one all-gather
                gl.copy_(vh, non_blocking=True)
                state["e2e_full"] = sdist.gather_features(gl, plan)

        dt = c.time_wall(e2e_step, ne)
        h2d = c.sum_over_ranks(float(n_have * 2))
        d2h = c.sum_over_ranks(float(n_local * rows * 8))
        # parity of the host path: the PCM16 host path must equal the device path run on the same (quantised) samples
        yq = (y16.to(c.dev).float() / 32768.0)
        chk = torch.empty((n_local, rows), dtype=torch.float64, device=c.dev)
        eng.segment_vectors_dev(yq.data_ptr(), units_l, p, ids, chk.data_ptr(), torch.cuda.current_stream().cuda_stream)
        same = bool(torch.equal(torch.nan_to_num(chk), torch.nan_to_num(vh.to(c.dev))))
        e2e = {"value": audio_total * ne / dt, "unit": w["unit"], "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "steps": ne, "ms_per_step": 1e3 * dt / ne, "input": "16-bit PCM mono in pinned host memory (the WAV payload)",
               "output": "float64 [segments, 24] vectors in pinned host memory" + (" + all-gather" if c.world > 1 else ""),
               "h2d_gbs_per_rank": (n_have * 2) / (dt / ne) / 1e9, "matches_device_path": same, "host_placement": c.placement}
        del yq, chk
        # the reference's own in-memory format for comparison: float32 samples in, same vectors out
        yh = torch.empty(n_have, dtype=torch.float32, pin_memory=True)
        yh.copy_(y)
        dt32 = c.time_wall(lambda: eng.segment_vectors_host(yh.data_ptr(), units_l, p, ids, out=vh_np), ne)
        e2e["f32"] = {"value": audio_total * ne / dt32, "unit": w["unit"], "h2d_bytes_per_step": int(c.sum_over_ranks(float(n_have * 4))),
                      "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * dt32 / ne}
        del yh, y16

    if c.rank == 0:
        # algorithmic bytes (SURVEY 8d): unique input samples + frame-feature rows, of THIS rank's block (one GPU against one peak)
        alg = 4.0 * (plan.seg_hop * n_local) + 4.0 * n_local * rows * T
        line = {
            "metric": w["metric"], "value": value, "unit": w["unit"], "n_gpus": c.world, "steps": args.steps, "warmup": c.warm,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"cfg4: {w['desc']}", "audio_hours": hours, "segments": plan.n_units, "segments_per_rank": n_local,
                       "rows": rows, "frames_per_segment": T, "aggregation": "mean",
                       "l2": "inputs larger than L2 (%.2f GB samples per rank per step)" % (n_have * 4 / 1e9),
                       "parallelism": f"segments block-partitioned over {c.world} GPU(s) with a {plan.seg_len - plan.seg_hop}-sample halo; "
                                      "one NCCL all-gather of the [segments, 24] float64 vectors inside the timed region"},
            "roofline": roofline_block(c, alg, prof, args.steps, ms, "frame_warp_kernel (framing+window+rFFT+fused feature epilogues)",
                                       c.traffic("cfg4"), {"finalize_ms_per_step": prof["finalize"][0] / args.steps,
                                                           "aggregate_ms_per_step": prof["other"][0] / args.steps}),
            "clocks": clk, "gpu_launches": int(sum(prof[k][1] for k in prof)), "checksum": checksum,
        }
        if gather_ms is not None:
            line["gather_ms"] = gather_ms
        if weak:
            line["weak"] = weak
        if e2e:
            line["e2e"] = e2e
    else:
        line = None
    return c.finish(line)


def shard(n, rank, world):
    base, extra = divmod(n, world)
    u0 = rank * base + min(rank, extra)
    return u0, u0 + base + (1 if rank < extra else 0)


def gather_block(c: Ctx, local, counts):
    """all-gather of per-rank blocks of equal trailing shape (padded to the largest count); returns the full block"""
    torch, dist = c.torch, c.dist
    if c.world == 1:
        return local
    mx = max(counts)
    pad = local
    if local.shape[0] != mx:
        pad = torch.zeros((mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
        pad[: local.shape[0]] = local
    buf = torch.empty((c.world * mx,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(buf, pad)
    return buf


def run_clips(c: Ctx):
    """cfg3: 100k one-second clips, MFCC13; clips block-partitioned over the ranks, feature block gathered inside the timed region."""
    from sygnals_b200 import _ffi
    from sygnals_b200.utils import synth
    torch, args, eng = c.torch, c.args, c.eng
    w = WORKLOADS[args.workload]
    sr, L = w["sr"], w["clip"]
    n_all = args.units or w["n_clips"]
    clip_s = L / float(sr)                                                # audio seconds per clip
    u0, u1 = shard(n_all, c.rank, c.world)
    n = u1 - u0
    counts = [shard(n_all, r, c.world)[1] - shard(n_all, r, c.world)[0] for r in range(c.world)]
    p = _ffi.make_params(eng.lib, sr, w["features"], w["fl"], w["hop"], feature_params=w["fp"])
    rows, T = eng.rows(p), eng.frame_count(L, w["fl"], w["hop"], True)
    y = torch.empty((n, L), dtype=torch.float32, device=c.dev)
    synth.torch_mixture_(y, sr, seed=77 + c.rank)
    out = torch.empty((n, rows, T), dtype=torch.float32, device=c.dev)
    units = eng.units_clips(n, L)
    stream = torch.cuda.current_stream().cuda_stream
    state = {}

    def step():
        eng.features_dev(y.data_ptr(), units, p, out.data_ptr(), stream)
        state["full"] = gather_block(c, out, counts)

    ms_max, ms, clk, prof = c.time_device(step, args.steps)
    c.dump({"features": state["full"]})                                 # float32 [clips, rows, frames]
    value = n_all * clip_s * args.steps / (ms_max * 1e-3)
    e2e = None
    if not args.no_e2e and args.workload == "cfg1":
        # the call a Sygnals user makes: extract_features(y float64, ...) -> DataFrame (H2D, kernels, D2H, float64 columns, pandas)
        import numpy as np
        from sygnals_b200.core.features import manager
        y64 = y[0].cpu().numpy().astype(np.float64)
        ne = max(3, args.e2e_steps)
        manager.extract_features(y64, sr, w["features"], frame_length=w["fl"], hop_length=w["hop"], feature_params=w["fp"])
        t0 = time.perf_counter()
        for _ in range(ne):
            df = manager.extract_features(y64, sr, w["features"], frame_length=w["fl"], hop_length=w["hop"], feature_params=w["fp"])
        dt = (time.perf_counter() - t0)
        e2e = {"value": clip_s * ne / dt, "unit": w["unit"], "h2d_bytes_per_step": int(L * 4), "d2h_bytes_per_step": int(out.numel() * 4),
               "steps": ne, "ms_per_step": 1e3 * dt / ne, "api": "sygnals_b200.core.features.manager.extract_features -> DataFrame",
               "columns": int(df.shape[1]), "frames": int(df.shape[0])}
    elif not args.no_e2e:
        # the clips as 16-bit PCM (what the dataset's WAV files hold) in pinned memory -> features in pinned memory
        y16 = torch.empty((n, L), dtype=torch.int16, pin_memory=True)
        y16.copy_((y * 32767.0).round().clamp(-32768, 32767).to(torch.int16))
        oh = torch.empty((n, rows, T), dtype=torch.float32, pin_memory=True)
        oh_np = oh.numpy()
        ne = max(1, min(args.steps, args.e2e_steps))
        dt = c.time_wall(lambda: eng.features_host_pcm(y16.data_ptr(), _ffi.PCM_S16, 1, units, p, out=oh_np), ne)
        yq = y16.to(c.dev).float() / 32768.0
        chk = torch.empty_like(out)
        eng.features_dev(yq.data_ptr(), units, p, chk.data_ptr(), stream)
        same = bool(torch.equal(oh.to(c.dev), chk))
        e2e = {"value": n_all * clip_s * ne / dt, "unit": w["unit"], "h2d_bytes_per_step": int(c.sum_over_ranks(float(n * L * 2))),
               "d2h_bytes_per_step": int(c.sum_over_ranks(float(out.numel() * 4))), "steps": ne, "ms_per_step": 1e3 * dt / ne,
               "input": "16-bit PCM clips in pinned host memory", "matches_device_path": same}
        del yq, chk, y16
        yh = torch.empty((n, L), dtype=torch.float32, pin_memory=True)
        yh.copy_(y)
        dt32 = c.time_wall(lambda: eng.features_host(None, units, p, out=oh_np, y_ptr=yh.data_ptr()), ne)
        e2e["f32"] = {"value": n_all * clip_s * ne / dt32, "unit": w["unit"], "h2d_bytes_per_step": int(c.sum_over_ranks(float(n * L * 4))),
                      "d2h_bytes_per_step": e2e["d2h_bytes_per_step"], "ms_per_step": 1e3 * dt32 / ne,
                      "matches_device_path": bool(torch.equal(oh.to(c.dev), out))}
    line = None
    if c.rank == 0:
        alg = 4.0 * n * L + 4.0 * out.numel()
        line = {"metric": w["metric"], "value": value, "unit": w["unit"], "n_gpus": c.world, "steps": args.steps, "warmup": c.warm,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"{args.workload}: {w['desc']}", "clips": n_all, "clips_per_rank": n, "rows": rows, "frames_per_clip": T,
                           "l2": ("inputs larger than L2 (%.2f GB per rank per step)" % (n * L * 4 / 1e9)) if n * L * 4 > (126 << 20)
                                 else "one clip (0.9 MB) stays in L2 between steps: this line is a LATENCY figure, not a bandwidth one",
                           "parallelism": f"clips block-partitioned over {c.world} GPU(s); all-gather of the feature block inside the timed region"},
                "roofline": roofline_block(c, alg, prof, args.steps, ms, f"frame_warp_kernel<n_fft {w['fl']}> (framing+window+rFFT+mel)",
                                           None, {"finalize_ms_per_step": prof["finalize"][0] / args.steps}),
                "clocks": clk, "gpu_launches": int(sum(prof[k][1] for k in prof))}
        if e2e:
            line["e2e"] = e2e
    return c.finish(line)


def run_stft(c: Ctx):
    """cfg2: STFT magnitude sweep over n_fft; one step = all six transforms of the clip batch."""
    from sygnals_b200 import _ffi
    from sygnals_b200.utils import synth
    torch, args, eng = c.torch, c.args, c.eng
    w = WORKLOADS["cfg2"]
    sr, L = w["sr"], w["clip"]
    n_all = args.units or w["n_clips"]
    u0, u1 = shard(n_all, c.rank, c.world)
    n = u1 - u0
    y = torch.empty((n, L), dtype=torch.float32, device=c.dev)
    synth.torch_mixture_(y, sr, seed=55 + c.rank)
    units = eng.units_clips(n, L)
    stream = torch.cuda.current_stream().cuda_stream
    sizes = [int(s) for s in args.nfft.split(",")] if args.nfft else CFG2_NFFT
    outs = {}
    for nf in sizes:
        T = eng.frame_count(L, nf, nf // 4, True)
        outs[nf] = torch.empty((n, nf // 2 + 1, T), dtype=torch.float32, device=c.dev)
    flush = torch.empty(192 << 20, dtype=torch.uint8, device=c.dev)    # > L2 (126 MB): the 0.26 GB input would otherwise stay hot between sizes

    def one(nf):
        eng.stft_dev(y.data_ptr(), units, nf, nf // 4, nf, 0, True, 0, _ffi.OUT_MAGNITUDE, outs[nf].data_ptr(), stream)

    peak, src = c.peaks()
    sweep, tot_ms, launches, clk_all = [], 0.0, 0, None
    for nf in sizes:
        def step(nf=nf):
            flush.zero_()
            one(nf)
        ms_max, ms, clk, prof = c.time_device(step, args.steps, sample_clocks=(nf == 2048 or len(sizes) == 1))
        k_ms, k_n = prof["frame"]
        clk_all = clk or clk_all
        alg = 4.0 * n * L + 4.0 * outs[nf].numel()
        ach = alg * args.steps / (k_ms * 1e-3) / 1e9
        sweep.append({"n_fft": nf, "kernel_ms": k_ms / args.steps, "achieved": ach, "frac": ach / peak, "algorithmic_bytes": alg,
                      "audio_s_per_s": c.world * n * args.steps / (c.max_over_ranks(k_ms) * 1e-3)})
        tot_ms += c.max_over_ranks(k_ms)
        launches += k_n
    c.dump({f"stft_magnitude_{nf}": outs[nf] for nf in sizes})          # float32 [clips, n_fft / 2 + 1, frames] per size
    value = n_all * len(sizes) * args.steps / (tot_ms * 1e-3)
    e2e = None
    if not args.no_e2e:
        yh = torch.empty((n, L), dtype=torch.float32, pin_memory=True)
        yh.copy_(y)
        import numpy as np
        ne = max(1, min(args.steps, args.e2e_steps))
        d2h = sum(outs[nf].numel() * 4 for nf in sizes)
        yh_np = yh.numpy().reshape(-1)
        ohs = {nf: torch.empty(tuple(outs[nf].shape), dtype=torch.float32, pin_memory=True) for nf in sizes}   # allocated once, reused

        def e2e_step():
            for nf in sizes:
                eng.stft_host(yh_np, units, nf, nf // 4, nf, 0, True, 0, _ffi.OUT_MAGNITUDE, out=ohs[nf].numpy())

        dt = c.time_wall(e2e_step, ne)
        e2e = {"value": n_all * len(sizes) * ne / dt, "unit": w["unit"], "h2d_bytes_per_step": int(c.sum_over_ranks(float(n * L * 4 * len(sizes)))),
               "d2h_bytes_per_step": int(c.sum_over_ranks(float(d2h))), "steps": ne, "ms_per_step": 1e3 * dt / ne,
               "matches_device_path": all(bool(torch.equal(ohs[nf].to(c.dev), outs[nf])) for nf in sizes)}
    line = None
    if c.rank == 0:
        worst = min(sweep, key=lambda s: s["frac"])
        line = {"metric": w["metric"], "value": value, "unit": w["unit"], "n_gpus": c.world, "steps": args.steps, "warmup": c.warm,
                "ms_per_step": tot_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"cfg2: {w['desc']}", "clips": n_all, "clips_per_rank": n, "n_fft": sizes,
                           "l2": "L2 flushed (192 MiB write) before every transform; the flush is outside the kernel's event pair",
                           "timing": "value and ms_per_step are sums of the STFT kernels' CUDA-event times (flush excluded)",
                           "parallelism": f"clips block-partitioned over {c.world} GPU(s), no collective"},
                "roofline": {"bound": "hbm", "kernel": "STFT kernels (framing+window+rFFT+|X|, transposed stores)", "achieved": worst["achieved"],
                             "peak": peak, "unit": "GB/s", "frac": worst["frac"], "peak_source": src, "traffic": None,
                             "which": f"the sweep's worst point (n_fft {worst['n_fft']})", "sweep": sweep},
                "clocks": clk_all, "gpu_launches": int(launches)}
        if e2e:
            line["e2e"] = e2e
    return c.finish(line)


def run_welch(c: Ctx):
    """cfg5: per (channel, second) Welch PSD + RMS + crest; channels block-partitioned over the ranks."""
    from sygnals_b200 import _ffi
    from sygnals_b200.utils import synth
    torch, args, eng = c.torch, c.args, c.eng
    w = WORKLOADS["cfg5"]
    sr = w["sr"]
    seconds = int(args.seconds or w["seconds"])
    c0, c1 = shard(w["channels"], c.rank, c.world)
    n = (c1 - c0) * seconds                                             # units of this rank: its channels' seconds
    n_all = w["channels"] * seconds
    y = torch.empty((n, sr), dtype=torch.float32, device=c.dev)
    synth.torch_mixture_(y, sr, seed=31 + c.rank)
    psd = torch.empty((n, 513), dtype=torch.float32, device=c.dev)
    st = torch.empty((n, 3), dtype=torch.float32, device=c.dev)
    units = eng.units_clips(n, sr)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        eng.psd_welch_dev(y.data_ptr(), units, float(sr), 0, 1024, 512, 1024, True, 0, psd.data_ptr(), st.data_ptr(), stream)

    ms_max, ms, clk, prof = c.time_device(step, args.steps)
    c.dump({"psd": psd, "stats": st})                                   # float32 [channel-seconds, 513] and [channel-seconds, 3]
    value = n_all * args.steps / (ms_max * 1e-3)
    e2e = None
    if not args.no_e2e:
        yh = torch.empty((n, sr), dtype=torch.float32, pin_memory=True)
        yh.copy_(y)
        ne = max(1, min(args.steps, args.e2e_steps))
        yh_np = yh.numpy().reshape(-1)
        dt = c.time_wall(lambda: eng.psd_welch_host(yh_np, units, float(sr), 0, 1024, 512, 1024, True, 0, stats=True), ne)
        e2e = {"value": n_all * ne / dt, "unit": w["unit"], "h2d_bytes_per_step": int(c.sum_over_ranks(float(n * sr * 4))),
               "d2h_bytes_per_step": int(c.sum_over_ranks(float(n * 516 * 4))), "steps": ne, "ms_per_step": 1e3 * dt / ne}
    line = None
    if c.rank == 0:
        alg = 4.0 * n * (sr + 515)
        line = {"metric": w["metric"], "value": value, "unit": w["unit"], "n_gpus": c.world, "steps": args.steps, "warmup": c.warm,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"cfg5: {w['desc']}", "seconds": seconds, "units": n_all, "units_per_rank": n,
                           "l2": "inputs larger than L2 (%.2f GB per rank per step)" % (n * sr * 4 / 1e9),
                           "parallelism": f"channels block-partitioned over {c.world} GPU(s), no collective"},
                "roofline": roofline_block(c, alg, prof, args.steps, ms, "welch"),
                "clocks": clk, "gpu_launches": int(sum(prof[k][1] for k in prof))}
        line["roofline"]["kernel"] = "welch_warp_kernel (detrend+window+rFFT+|X|^2 averaged over 49 sub-segments, unit RMS/crest)"
        if e2e:
            line["e2e"] = e2e
    return c.finish(line)


def run_native(args):
    c = Ctx(args)
    kind = WORKLOADS[args.workload]["kind"]
    return {"segments": run_segments, "clips": run_clips, "stft": run_stft, "welch": run_welch}[kind](c)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--hours", type=float, default=0.0, help="cfg4: audio hours of the recording (default 10)")
    ap.add_argument("--units", type=int, default=0, help="cfg3 / cfg2: number of clips (default: the workload's)")
    ap.add_argument("--seconds", type=int, default=0, help="cfg5: seconds per channel (default 600)")
    ap.add_argument("--nfft", default="", help="cfg2: comma-separated subset of the sweep")
    ap.add_argument("--ws-mb", type=int, default=0, help="engine workspace limit in MiB (0: library default)")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="cfg4: skip the weak-scaling side measurement")
    ap.add_argument("--cpu-units", type=int, default=0, help="units per step of the CPU reference arm")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="native arm: write the outputs of the last timed step as DIR/<name>.npy (under 64 MB in all: a seeded sample of a larger "
                         "output); cfg4/cfg1/cfg3 write the output gathered from all ranks, cfg2/cfg5 rank 0's block"),
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs")
    guard_stdout()
    if args.impl == "reference":
        return run_reference(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
