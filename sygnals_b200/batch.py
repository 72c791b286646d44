"""Additive batched entry points of the B200 engine (the reference has none: it loops over files / segments in Python).

* :func:`extract_features_batch`  -- many equal-length clips in one launch (BASELINE cfg3 shape)
* :func:`segment_features`        -- ``segment_fixed_length`` + ``extract_features`` per segment fused into one launch over
                                     the un-segmented recording (BASELINE cfg4 shape); segments are framed by index
* :func:`extract_features_ragged`, :func:`clip_vectors`
                                  -- clips of different lengths (a folder of files, variable-length segments) in one launch,
                                     each clip framed on its own: no padding to the longest
* :func:`stft_batch`, :func:`psd_welch_batch`

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
            names += [f"mfcc_{i}" for i in range(int(fp.get("mfcc", {}).get("n_mfcc", 13)))]
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
    p = _ffi.make_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
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
    total = int(y.shape[0])
    seg_len, seg_hop, starts, valid = eng.lib.segment_table(total, sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec)
    p = _ffi.make_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
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
    out = _run(y, units, n, p, eng)
    # `keep` (device tables) may be dropped without a host synchronisation: the kernels are queued on the current torch stream and
    # the caching allocator reuses a freed block only for work queued later on that stream
    del keep
    return {"names": feature_row_names(features, feature_params), "features": out, "starts": starts, "valid": valid,
            "seg_len": seg_len, "seg_hop": seg_hop}


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
    p = _ffi.make_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
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
