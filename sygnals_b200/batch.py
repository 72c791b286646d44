"""Additive batched entry points of the B200 engine (the reference has none: it loops over files / segments in Python).

* :func:`extract_features_batch`  -- many equal-length clips in one launch (BASELINE cfg3 shape)
* :func:`segment_features`        -- ``segment_fixed_length`` + ``extract_features`` per segment fused into one launch over
                                     the un-segmented recording (BASELINE cfg4 shape); segments are framed by index
* :func:`extract_features_ragged`, :func:`clip_vectors`
                                  -- clips of different lengths (a folder of files, variable-length segments) in one launch,
                                     each clip framed on its own: no padding to the longest
* :func:`mel_spectrogram_batch`, :func:`segment_mel_spectrogram`, :func:`mel_spectrogram_ragged`
                                  -- the (log-)mel spectrogram ``extract_features`` computes for its MFCCs, per clip or segment,
                                     for the same three input shapes
* :func:`stft_batch`, :func:`psd_welch_batch`
* :func:`channel_psd`, :func:`channel_vectors`
                                  -- per-channel Welch PSDs / segment vectors of a multi-channel PCM recording (a WAV file or
                                     a :class:`Payload`, BASELINE cfg5 shape): the interleaved bytes cross PCIe as they are and
                                     are de-interleaved on the device

Inputs may be numpy arrays (host path: chunked H2D / kernels / D2H inside the library) or CUDA ``torch`` tensors (device
path: asynchronous on the current torch stream, result stays in HBM).  Row naming follows manager.py:337-343,365-369.
"""
from __future__ import annotations

from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from . import _ffi


def feature_row_names(features: Sequence[str], feature_params: Optional[dict] = None) -> List[str]:
    fp = feature_params or {}
    names: List[str] = []
    for f in features:
        if f == "mfcc":
            names += [f"mfcc_{i}" for i in range(_ffi.mfcc_count(fp))]
        elif f == "spectral_contrast":
            nb = int(fp.get("spectral_contrast", {}).get("n_bands", 6))
            names += [f"contrast_band_{i}" for i in range(nb)] + ["contrast_delta"]
        else:
            names.append(f)
    return names


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _run(y, units_fn, n_units, p, eng):
    rows = eng.rows(p)
    T = eng.frame_count(units_fn.unit_len, p.frame_length, p.hop_length, p.center)
    if _is_torch(y):
        import torch
        if not y.is_cuda:
            raise ValueError("torch inputs must live on a CUDA device (use numpy arrays for host data)")
        if y.dtype != torch.float32 or not y.is_contiguous():
            y = y.contiguous().float()
        out = torch.empty((n_units, rows, T), dtype=torch.float32, device=y.device)
        if out.numel():
            eng.features_dev(y.data_ptr(), units_fn, p, out.data_ptr(), torch.cuda.current_stream(y.device).cuda_stream)
        return out
    return eng.features_host(np.ascontiguousarray(y, dtype=np.float32).reshape(-1), units_fn, p)


def _engine_for(y, device):
    if _is_torch(y) and y.is_cuda:
        return _ffi.engine(y.device.index if y.device.index is not None else 0)
    return _ffi.engine(device)


def extract_features_batch(clips, sr: int, features: Sequence[str], frame_length: int = 2048, hop_length: int = 512,
                           center: bool = True, window: str = "hann", feature_params: Optional[dict] = None,
                           device: Optional[int] = None) -> Tuple[List[str], "np.ndarray"]:
    """``clips``: ``[n_clips, L]`` float32 (numpy or CUDA torch).  Returns (row names, float32 ``[n_clips, rows, T]``);
    clip ``c`` gets exactly what ``extract_features(clips[c], ...)`` returns (per-clip ``ref=np.max`` in power_to_db)."""
    if clips.ndim != 2:
        raise ValueError("clips must be a 2D array [n_clips, n_samples].")
    eng = _engine_for(clips, device)
    p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
    n, L = int(clips.shape[0]), int(clips.shape[1])
    out = _run(clips, eng.units_clips(n, L), n, p, eng)
    return feature_row_names(features, feature_params), out


def segment_features(y, sr: int, segment_length_sec: float, features: Sequence[str], overlap_ratio: float = 0.0, pad: bool = True,
                     min_segment_length_sec: Optional[float] = None, frame_length: int = 2048, hop_length: int = 512,
                     center: bool = True, window: str = "hann", feature_params: Optional[dict] = None,
                     device: Optional[int] = None) -> Dict[str, object]:
    """One launch over a whole recording: segment boundaries by ``segment_fixed_length`` arithmetic
    (segmentation.py:62-114), zero-padded tail by predicate, per-segment features as ``extract_features`` on each segment.
    Returns {'names', 'features' [n_seg, rows, T], 'starts', 'valid', 'seg_len', 'seg_hop'}."""
    if y.ndim != 1:
        raise ValueError("Input signal y must be 1D.")
    eng = _engine_for(y, device)
    seg = _segments(eng, y, sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec)
    p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
    out = _run(y, seg.units, len(seg.starts), p, eng)
    return {"names": feature_row_names(features, feature_params), "features": out, "starts": seg.starts, "valid": seg.valid,
            "seg_len": seg.seg_len, "seg_hop": seg.seg_hop}


class _Segments(NamedTuple):
    units: object                   # _ffi.SygUnits
    keep: object                    # the tables `units` points at
    starts: np.ndarray
    valid: np.ndarray
    seg_len: int
    seg_hop: int


def _segments(eng, y, sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec) -> _Segments:
    """The units of ``segment_fixed_length`` over the 1-D recording ``y``: analytic starts when they are multiples of the hop, else
    the segment table (on ``y``'s device for a CUDA tensor).  The tables may be dropped without a host synchronisation once the
    call is queued: the kernels run on the current torch stream, and the caching allocator reuses a freed block only for work queued
    later on that stream."""
    total = int(y.shape[0])
    seg_len, seg_hop, starts, valid = eng.lib.segment_table(total, sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec)
    n = len(starts)
    analytic = n > 0 and min_segment_length_sec is None and bool((starts == np.arange(n, dtype=np.int64) * seg_hop).all())
    if n == 0 or analytic:
        units = eng.units_clips(n, seg_len, total_len=total, stride=seg_hop)
        keep = None
    elif _is_torch(y):
        import torch
        st = torch.from_numpy(starts).to(y.device)
        va = torch.from_numpy(valid).to(y.device)
        units = eng.units_table(st.data_ptr(), va.data_ptr(), n, seg_len, total)
        keep = (st, va)
    else:
        units = eng.units_table(starts.ctypes.data, valid.ctypes.data, n, seg_len, total)
        keep = (starts, valid)
    return _Segments(units, keep, starts, valid, seg_len, seg_hop)


class Windows(NamedTuple):
    """Windows of ONE sample buffer as ragged clips, without a copy: clip ``u`` is ``y[starts[u] : starts[u] + lengths[u]]``
    (windows may overlap or leave gaps; e.g. the variable-length segments of one recording).  ``y``: 1-D float32 numpy array or
    CUDA tensor; ``starts`` / ``lengths``: integer sequences (numpy, lists or torch tensors on any device)."""
    y: object
    starts: object
    lengths: object


def _int_table(t) -> np.ndarray:
    if _is_torch(t):
        t = t.detach().cpu().numpy()
    a = np.asarray(t)
    if a.size and a.dtype.kind not in "iu":
        raise ValueError("starts and lengths must be integers")
    return a.astype(np.int64).reshape(-1)


def _ragged_input(clips):
    """``clips`` -> (y, starts, lengths).  A :class:`Windows` is taken as it is; anything else is a sequence of 1-D clips, concatenated
    once (numpy arrays -> host path, CUDA tensors -> device path)."""
    if isinstance(clips, Windows):
        if getattr(clips.y, "ndim", None) != 1:
            raise ValueError("Windows.y must be a 1-D sample buffer")
        starts, lengths = _int_table(clips.starts), _int_table(clips.lengths)
        if starts.shape != lengths.shape:
            raise ValueError("Windows.starts and Windows.lengths must have the same length")
        return clips.y, starts, lengths
    clips = list(clips)
    for c in clips:
        if getattr(c, "ndim", None) != 1:
            raise ValueError("every clip must be a 1-D array (use batch.Windows for windows of one buffer)")
    lengths = np.array([int(c.shape[0]) for c in clips], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64) if len(clips) else np.zeros(0, dtype=np.int64)
    if clips and all(_is_torch(c) for c in clips):
        import torch
        if not all(c.is_cuda for c in clips):
            raise ValueError("torch inputs must live on a CUDA device (use numpy arrays for host data)")
        return torch.cat([c.float() for c in clips]), starts, lengths
    if any(_is_torch(c) for c in clips):
        raise ValueError("clips must be all numpy arrays or all CUDA tensors")
    y = np.concatenate([np.asarray(c, dtype=np.float32) for c in clips]) if clips else np.zeros(0, dtype=np.float32)
    return y, starts, lengths


def _ragged_call(clips, sr, features, frame_length, hop_length, center, window, feature_params, device, agg=None):
    y, starts, lengths = _ragged_input(clips)
    if getattr(y, "ndim", None) != 1:
        raise ValueError("the sample buffer must be 1-D")
    eng = _engine_for(y, device)
    p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
    units = eng.ragged_units(starts, lengths, int(y.shape[0]))
    names = feature_row_names(features, feature_params)
    ids = None
    if agg is not None:
        from .core.ml_utils.formatters import _agg_ids
        ids = _agg_ids(names, agg)
    foff = eng.lib.ragged_frame_offsets(units, frame_length, hop_length, center)
    rows = eng.rows(p)
    if _is_torch(y):
        import torch
        if not y.is_cuda:
            raise ValueError("torch inputs must live on a CUDA device (use numpy arrays for host data)")
        if y.dtype != torch.float32 or not y.is_contiguous():
            y = y.contiguous().float()
        stream = torch.cuda.current_stream(y.device).cuda_stream
        if ids is None:
            out = torch.empty((rows, int(foff[-1])), dtype=torch.float32, device=y.device)
            eng.features_ragged_dev(y.data_ptr(), units, p, out.data_ptr(), stream)
        else:
            out = torch.empty((len(lengths), rows), dtype=torch.float64, device=y.device)
            eng.segment_vectors_ragged_dev(y.data_ptr(), units, p, ids, out.data_ptr(), stream)
    else:
        y = np.ascontiguousarray(y, dtype=np.float32)
        out = eng.features_ragged_host(y, units, p) if ids is None else eng.segment_vectors_ragged_host(y, units, p, ids)
    return names, out, foff


def extract_features_ragged(clips, sr: int, features: Sequence[str], frame_length: int = 2048, hop_length: int = 512,
                            center: bool = True, window: str = "hann", feature_params: Optional[dict] = None,
                            device: Optional[int] = None) -> Dict[str, object]:
    """Clips of different lengths in one launch.  ``clips``: a sequence of 1-D arrays (numpy: host path; CUDA tensors: device path,
    asynchronous on the current stream) or a :class:`Windows` ``(y, starts, lengths)`` addressing windows of one buffer without a copy.
    Returns {'names', 'features': float32 ``[rows, F]``, 'frame_offsets': int64 ``[n_clips + 1]``}: columns
    ``frame_offsets[c] .. frame_offsets[c + 1] - 1`` are exactly ``extract_features(clip c, ...)`` (the layout of
    ``format_feature_vectors_per_segment``'s features_dict with those ranges as segment indices)."""
    names, out, foff = _ragged_call(clips, sr, features, frame_length, hop_length, center, window, feature_params, device)
    return {"names": names, "features": out, "frame_offsets": foff}


def clip_vectors(clips, sr: int, features: Sequence[str], aggregation="mean", frame_length: int = 2048, hop_length: int = 512,
                 center: bool = True, window: str = "hann", feature_params: Optional[dict] = None, device: Optional[int] = None):
    """One vector per clip: ``extract_features`` per clip followed by ``format_feature_vectors_per_segment`` with every clip as one
    segment.  ``clips`` as in :func:`extract_features_ragged`; ``aggregation`` a name or a per-row dict (formatters.py:39-45).
    Returns (row names, float64 ``[n_clips, rows]``); a clip without frames gives a NaN row."""
    names, out, _ = _ragged_call(clips, sr, features, frame_length, hop_length, center, window, feature_params, device, agg=aggregation)
    return names, out


def _mel_params(lib, sr, frame_length, hop_length, center, window, n_mels, fmin, fmax, power):
    """The mel stage's arguments (manager.py:213-217) as a parameter block without features.  Invalid values raise ValueError;
    what the kernels do not serve (n_mels above 256, transform lengths, windows) raises NotImplementedError from the library."""
    if int(hop_length) < 1:
        raise ValueError(f"hop_length={hop_length} must be >= 1")
    if int(n_mels) < 1:
        raise ValueError(f"n_mels={n_mels} must be positive")
    if not float(power) > 0:
        raise ValueError(f"power={power} must be positive")
    top = sr / 2.0 if fmax is None else float(fmax)
    if not top > float(fmin):
        raise ValueError(f"fmax={top} must be above fmin={fmin}")
    mel = {"n_mels": int(n_mels), "fmin": float(fmin), "fmax": fmax, "power": float(power)}
    return _ffi.make_params(lib, sr, [], frame_length, hop_length, center, window, {"mfcc": mel})


def _run_mel(y, units, p, db, eng):
    T = eng.frame_count(units.unit_len, p.frame_length, p.hop_length, p.center)
    if _is_torch(y):
        import torch
        if not y.is_cuda:
            raise ValueError("torch inputs must live on a CUDA device (use numpy arrays for host data)")
        if y.dtype != torch.float32 or not y.is_contiguous():
            y = y.contiguous().float()
        out = torch.empty((int(units.n_units), int(p.n_mels), T), dtype=torch.float32, device=y.device)
        eng.mel_spectrogram_dev(y.data_ptr(), units, p, db, out.data_ptr(), torch.cuda.current_stream(y.device).cuda_stream)
        return out
    return eng.mel_spectrogram_host(np.ascontiguousarray(y, dtype=np.float32).reshape(-1), units, p, db)


def mel_spectrogram_batch(clips, sr: int, frame_length: int = 2048, hop_length: int = 512, center: bool = True, window: str = "hann",
                          n_mels: int = 128, fmin: float = 0.0, fmax: Optional[float] = None, power: float = 2.0, db: bool = True,
                          device: Optional[int] = None):
    """``clips``: ``[n_clips, L]`` float32 (numpy: host path; CUDA torch: asynchronous on the current stream).  Returns float32
    ``[n_clips, n_mels, T]``: per clip the mel spectrogram ``extract_features`` builds for its MFCCs (manager.py:213-223),
    ``power_to_db(S_mel, ref=np.max)`` (clip's own maximum, top_db 80) with ``db``, ``S_mel`` without."""
    if clips.ndim != 2:
        raise ValueError("clips must be a 2D array [n_clips, n_samples].")
    eng = _engine_for(clips, device)
    p = _mel_params(eng.lib, sr, frame_length, hop_length, center, window, n_mels, fmin, fmax, power)
    return _run_mel(clips, eng.units_clips(int(clips.shape[0]), int(clips.shape[1])), p, db, eng)


def segment_mel_spectrogram(y, sr: int, segment_length_sec: float, overlap_ratio: float = 0.0, pad: bool = True,
                            min_segment_length_sec: Optional[float] = None, frame_length: int = 2048, hop_length: int = 512,
                            center: bool = True, window: str = "hann", n_mels: int = 128, fmin: float = 0.0, fmax: Optional[float] = None,
                            power: float = 2.0, db: bool = True, device: Optional[int] = None) -> Dict[str, object]:
    """:func:`mel_spectrogram_batch` of every segment of one recording, segmented as :func:`segment_features` does (one launch over
    the un-segmented recording).  Returns {'mel' ``[n_seg, n_mels, T]``, 'starts', 'valid', 'seg_len', 'seg_hop'}."""
    if y.ndim != 1:
        raise ValueError("Input signal y must be 1D.")
    eng = _engine_for(y, device)
    seg = _segments(eng, y, sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec)
    p = _mel_params(eng.lib, sr, frame_length, hop_length, center, window, n_mels, fmin, fmax, power)
    out = _run_mel(y, seg.units, p, db, eng)
    return {"mel": out, "starts": seg.starts, "valid": seg.valid, "seg_len": seg.seg_len, "seg_hop": seg.seg_hop}


def mel_spectrogram_ragged(clips, sr: int, frame_length: int = 2048, hop_length: int = 512, center: bool = True, window: str = "hann",
                           n_mels: int = 128, fmin: float = 0.0, fmax: Optional[float] = None, power: float = 2.0, db: bool = True,
                           device: Optional[int] = None) -> Dict[str, object]:
    """Mel spectrograms of clips of different lengths in one launch; ``clips`` as in :func:`extract_features_ragged`.  Returns
    {'mel': float32 ``[n_mels, F]``, 'frame_offsets': int64 ``[n_clips + 1]``}: columns ``frame_offsets[c] ..
    frame_offsets[c + 1] - 1`` are :func:`mel_spectrogram_batch` of clip c alone."""
    y, starts, lengths = _ragged_input(clips)
    if getattr(y, "ndim", None) != 1:
        raise ValueError("the sample buffer must be 1-D")
    eng = _engine_for(y, device)
    p = _mel_params(eng.lib, sr, frame_length, hop_length, center, window, n_mels, fmin, fmax, power)
    units = eng.ragged_units(starts, lengths, int(y.shape[0]))
    foff = eng.lib.ragged_frame_offsets(units, frame_length, hop_length, center)
    if _is_torch(y):
        import torch
        if not y.is_cuda:
            raise ValueError("torch inputs must live on a CUDA device (use numpy arrays for host data)")
        if y.dtype != torch.float32 or not y.is_contiguous():
            y = y.contiguous().float()
        out = torch.empty((int(n_mels), int(foff[-1])), dtype=torch.float32, device=y.device)
        eng.mel_spectrogram_ragged_dev(y.data_ptr(), units, p, db, out.data_ptr(), torch.cuda.current_stream(y.device).cuda_stream)
    else:
        out = eng.mel_spectrogram_ragged_host(np.ascontiguousarray(y, dtype=np.float32), units, p, db)
    return {"mel": out, "frame_offsets": foff}


def stft_batch(clips, n_fft: int = 2048, hop_length: Optional[int] = None, win_length: Optional[int] = None, window: str = "hann",
               center: bool = True, pad_mode: str = "constant", output: str = "magnitude", device: Optional[int] = None):
    """``[n_clips, L]`` -> ``[n_clips, 1 + n_fft/2, T]`` complex64 / float32 magnitude / float32 power (BASELINE cfg2)."""
    if clips.ndim != 2:
        raise ValueError("clips must be a 2D array [n_clips, n_samples].")
    kinds = {"complex": _ffi.OUT_COMPLEX, "magnitude": _ffi.OUT_MAGNITUDE, "power": _ffi.OUT_POWER}
    if output not in kinds:
        raise ValueError(f"output must be one of {sorted(kinds)}")
    win_length = n_fft if win_length is None else win_length
    hop_length = win_length // 4 if hop_length is None else hop_length
    if window.lower() not in _ffi.WINDOW_IDS:
        raise NotImplementedError(f"window={window!r}")
    if pad_mode not in _ffi.PAD_IDS:
        raise NotImplementedError(f"pad_mode={pad_mode!r}")
    eng = _engine_for(clips, device)
    n, L = int(clips.shape[0]), int(clips.shape[1])
    units = eng.units_clips(n, L)
    wid, pid = _ffi.WINDOW_IDS[window.lower()], _ffi.PAD_IDS[pad_mode]
    if _is_torch(clips):
        import torch
        y = clips if (clips.dtype == torch.float32 and clips.is_contiguous()) else clips.contiguous().float()
        T = eng.frame_count(L, n_fft, hop_length, center)
        dt = torch.complex64 if output == "complex" else torch.float32
        out = torch.empty((n, 1 + n_fft // 2, T), dtype=dt, device=y.device)
        if out.numel():
            eng.stft_dev(y.data_ptr(), units, n_fft, hop_length, win_length, wid, center, pid, kinds[output], out.data_ptr(),
                         torch.cuda.current_stream(y.device).cuda_stream)
        return out
    return eng.stft_host(np.ascontiguousarray(clips, dtype=np.float32).reshape(-1), units, n_fft, hop_length, win_length, wid,
                         center, pid, kinds[output])


def psd_welch_batch(windows, fs: float, nperseg: int = 1024, noverlap: Optional[int] = None, nfft: Optional[int] = None,
                    window: str = "hann", detrend: bool = True, scaling: str = "density", stats: bool = True,
                    device: Optional[int] = None):
    """``[n_units, L]`` (e.g. channel-seconds, BASELINE cfg5) -> (psd ``[n_units, 1 + nfft/2]``, stats ``[n_units, 3]`` =
    rms, crest factor, peak of each unit)."""
    if windows.ndim != 2:
        raise ValueError("windows must be a 2D array [n_units, n_samples].")
    eng = _engine_for(windows, device)
    n, L = int(windows.shape[0]), int(windows.shape[1])
    nfft = nperseg if nfft is None else nfft
    noverlap = nperseg // 2 if noverlap is None else noverlap
    wid, sid = _ffi.WINDOW_IDS[window.lower()], _ffi.SCALING_IDS[scaling]
    units = eng.units_clips(n, L)
    if _is_torch(windows):
        import torch
        y = windows if (windows.dtype == torch.float32 and windows.is_contiguous()) else windows.contiguous().float()
        psd = torch.empty((n, 1 + nfft // 2), dtype=torch.float32, device=y.device)
        st = torch.empty((n, 3), dtype=torch.float32, device=y.device) if stats else None
        if n:
            eng.psd_welch_dev(y.data_ptr(), units, fs, wid, nperseg, noverlap, nfft, detrend, sid, psd.data_ptr(),
                              st.data_ptr() if stats else 0, torch.cuda.current_stream(y.device).cuda_stream)
        return (psd, st) if stats else psd
    return eng.psd_welch_host(np.ascontiguousarray(windows, dtype=np.float32).reshape(-1), units, fs, wid, nperseg, noverlap, nfft,
                              detrend, sid, stats=stats)


class Payload(NamedTuple):
    """An interleaved PCM payload in host memory: ``raw`` the bytes (a numpy array or any buffer), ``fmt`` one of ``_ffi.PCM_*``,
    ``channels`` samples per frame, ``sample_rate`` in Hz."""
    raw: object
    fmt: int
    channels: int
    sample_rate: int


def _pcm_source(source):
    """(uint8 array, fmt, channels, frames, sample_rate) of a WAV path (memory-mapped payload) or a :class:`Payload`."""
    if isinstance(source, Payload):
        if _is_torch(source.raw):
            raise ValueError("Payload.raw must be host memory (numpy array or buffer)")
        raw = source.raw if isinstance(source.raw, np.ndarray) else np.frombuffer(source.raw, dtype=np.uint8)
        raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
        fmt, ch, sr = int(source.fmt), int(source.channels), int(source.sample_rate)
        if fmt not in _ffi.PCM_BYTES:
            raise ValueError(f"unknown PCM sample format {fmt}")
        if not 1 <= ch <= 64:
            raise ValueError(f"channels={ch}: supported range is [1, 64]")
        return raw, fmt, ch, raw.size // (ch * _ffi.PCM_BYTES[fmt]), sr
    from .core.audio import io as sio
    info = sio.wav_info(source)
    raw, frames = sio.wav_payload(info)
    return raw, info.fmt, info.channels, frames, info.sample_rate


def channel_psd(source, window_sec: float = 1.0, overlap_ratio: float = 0.0, pad: bool = True, nperseg: int = 1024,
                noverlap: Optional[int] = None, nfft: Optional[int] = None, window: str = "hann", detrend: bool = True,
                scaling: str = "density", stats: bool = True, device: Optional[int] = None) -> Dict[str, object]:
    """Welch PSD per (window, channel) of a multi-channel PCM recording (BASELINE cfg5: a machinery monitor's WAV / DAQ payload).
    ``source``: a WAV path (memory-mapped) or a :class:`Payload` in host memory.  Windows follow ``segment_fixed_length``
    (segmentation.py:62-114) over the frames; each (window, channel) is ``compute_psd_welch`` of that channel's samples.
    Returns {'freqs', 'psd' float32 ``[n_windows, channels, 1 + nfft/2]``, 'stats' float32 ``[n_windows, channels, 3]`` (rms, crest
    factor, peak; None without ``stats``), 'starts', 'valid', 'sample_rate'}."""
    raw, fmt, ch, frames, sr = _pcm_source(source)
    eng = _ffi.engine(device)
    seg_len, _, starts, valid = eng.lib.segment_table(frames, sr, window_sec, overlap_ratio, pad)
    nfft = nperseg if nfft is None else nfft
    noverlap = nperseg // 2 if noverlap is None else noverlap
    if window.lower() not in _ffi.WINDOW_IDS:
        raise NotImplementedError(f"window={window!r}")
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, len(starts), seg_len, frames)
    res = eng.psd_welch_host_pcm_channels(raw.ctypes.data, fmt, ch, units, sr, _ffi.WINDOW_IDS[window.lower()], nperseg, noverlap,
                                          nfft, detrend, _ffi.SCALING_IDS[scaling], stats=stats)
    psd, st = res if stats else (res, None)
    return {"freqs": np.fft.rfftfreq(nfft, d=1.0 / sr), "psd": psd, "stats": st, "starts": starts, "valid": valid, "sample_rate": sr}


def channel_vectors(source, segment_length_sec: float, features: Sequence[str], aggregation="mean", overlap_ratio: float = 0.0,
                    pad: bool = True, frame_length: int = 2048, hop_length: int = 512, center: bool = True, window: str = "hann",
                    feature_params: Optional[dict] = None, device: Optional[int] = None):
    """One vector per (segment, channel) of a multi-channel PCM recording: ``extract_features`` per segment of each channel followed
    by ``format_feature_vectors_per_segment`` (``aggregation`` a name or a per-row dict, formatters.py:39-45).  ``source`` as in
    :func:`channel_psd`.  Returns (row names, float64 ``[n_segments, channels, rows]``)."""
    raw, fmt, ch, frames, sr = _pcm_source(source)
    eng = _ffi.engine(device)
    seg_len, _, starts, valid = eng.lib.segment_table(frames, sr, segment_length_sec, overlap_ratio, pad)
    p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
    names = feature_row_names(features, feature_params)
    from .core.ml_utils.formatters import _agg_ids
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, len(starts), seg_len, frames)
    return names, eng.segment_vectors_host_pcm_channels(raw.ctypes.data, fmt, ch, units, p, _agg_ids(names, aggregation))
