"""Audio ingest of the B200 engine: the step in front of the segment->features path.

Mirror of ``sygnals/core/audio/io.py:38-102`` (``load_audio`` -> ``librosa.load`` -> ``soundfile.read(dtype='float32')`` +
``librosa.to_mono``) for RIFF/WAVE files.  The header is parsed here on the host; the payload (the bytes of the ``data`` chunk)
goes to the GPU as it lies in the file and ``libsygb200`` de-interleaves, normalises and mixes it down there
(``syg_ingest_pcm`` / ``syg_features_host_pcm`` / ``syg_segment_vectors_host_pcm``), or keeps one plane per channel
(``syg_ingest_pcm_channels`` for ``mono=False``), so a 16-bit recording crosses PCIe at 2 bytes per sample instead of the
reference's 8 (float64).

Not served here (they stay on the reference path): compressed formats, and resampling (``sr`` different from the file's rate).
"""
from __future__ import annotations

import os
import struct
from dataclasses import dataclass
from pathlib import Path
from typing import Optional, Tuple, Union

import numpy as np

from ... import _ffi

WAVE_FORMAT_PCM, WAVE_FORMAT_IEEE_FLOAT, WAVE_FORMAT_EXTENSIBLE = 0x0001, 0x0003, 0xFFFE


@dataclass
class WavInfo:
    """Layout of a WAV file's sample payload."""
    path: str
    sample_rate: int
    channels: int
    fmt: int                 # _ffi.PCM_*
    data_offset: int         # byte offset of the first frame in the file
    n_frames: int            # frames (= samples per channel)

    @property
    def frame_bytes(self) -> int:
        return self.channels * _ffi.PCM_BYTES[self.fmt]


def wav_info(path: Union[str, os.PathLike]) -> WavInfo:
    """Parse the RIFF chunks of a WAV file (PCM 8/16/24/32 bit or IEEE float32, plain or WAVE_FORMAT_EXTENSIBLE)."""
    path = os.fspath(path)
    size = os.path.getsize(path)
    with open(path, "rb") as f:
        head = f.read(12)
        if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
            raise ValueError(f"{path}: not a RIFF/WAVE file")
        fmt_tag = channels = sr = bits = None
        pos = 12
        while pos + 8 <= size:
            f.seek(pos)
            cid, clen = struct.unpack("<4sI", f.read(8))
            body = pos + 8
            if cid == b"fmt ":
                raw = f.read(min(clen, 40))
                if len(raw) < 16:
                    raise ValueError(f"{path}: truncated fmt chunk")
                fmt_tag, channels, sr, _, _, bits = struct.unpack("<HHIIHH", raw[:16])
                if fmt_tag == WAVE_FORMAT_EXTENSIBLE and len(raw) >= 26:
                    fmt_tag = struct.unpack("<H", raw[24:26])[0]          # first two bytes of the SubFormat GUID
            elif cid == b"data":
                if fmt_tag is None:
                    raise ValueError(f"{path}: data chunk before fmt chunk")
                clen = min(clen, size - body)                              # streamed files carry 0xFFFFFFFF / stale lengths
                if fmt_tag == WAVE_FORMAT_PCM and bits in (8, 16, 24, 32):
                    fmt = {8: _ffi.PCM_U8, 16: _ffi.PCM_S16, 24: _ffi.PCM_S24, 32: _ffi.PCM_S32}[bits]
                elif fmt_tag == WAVE_FORMAT_IEEE_FLOAT and bits == 32:
                    fmt = _ffi.PCM_F32
                else:
                    raise NotImplementedError(f"{path}: WAV format tag {fmt_tag:#x} with {bits} bits has no ingest kernel")
                if not channels or channels > 64:
                    raise NotImplementedError(f"{path}: {channels} channels")
                fb = channels * _ffi.PCM_BYTES[fmt]
                return WavInfo(path, int(sr), int(channels), fmt, body, clen // fb)
            pos = body + clen + (clen & 1)                                 # chunks are word aligned
    raise ValueError(f"{path}: no data chunk")


def wav_payload(info: WavInfo, offset: float = 0.0, duration: Optional[float] = None) -> Tuple[np.ndarray, int]:
    """Memory map of the payload bytes for ``[offset, offset + duration)`` seconds (librosa.load's frame arithmetic:
    ``start = int(offset * sr)``, ``frames = int(duration * sr)``).  Returns (uint8 array, frames)."""
    start = min(int(offset * info.sample_rate), info.n_frames) if offset else 0
    frames = info.n_frames - start
    if duration is not None:
        frames = max(0, min(frames, int(duration * info.sample_rate)))
    fb = info.frame_bytes
    if frames == 0:
        return np.zeros(0, dtype=np.uint8), 0
    mm = np.memmap(info.path, dtype=np.uint8, mode="r", offset=info.data_offset + start * fb, shape=(frames * fb,))
    return mm, frames


def load_audio(file_path: Union[str, os.PathLike], sr: Optional[int] = None, mono: bool = True, offset: float = 0.0,
               duration: Optional[float] = None, device: Optional[int] = None) -> Tuple[np.ndarray, int]:
    """``load_audio`` of the reference (io.py:38-102) for WAV files: float64 samples in [-1, 1) and the sample rate.
    The payload is widened and mixed down on the GPU; values are identical to soundfile's float32 read followed by
    ``np.mean(axis=0)``."""
    p = Path(file_path)
    if not p.exists():
        raise FileNotFoundError(f"Audio input file not found: {p}")
    if not p.is_file():
        raise ValueError(f"Input path is not a file: {p}")
    info = wav_info(p)
    if sr is not None and int(sr) != info.sample_rate:
        raise NotImplementedError(f"sr={sr}: resampling (native rate {info.sample_rate}) stays on the reference path")
    raw, frames = wav_payload(info, offset, duration)
    if not mono and info.channels > 1:
        # (n_channels, n_samples) like librosa
        return pcm_to_planes(raw, info.fmt, info.channels, device).astype(np.float64), info.sample_rate
    return pcm_to_mono(raw, info.fmt, info.channels, device).astype(np.float64), info.sample_rate


def pcm_to_mono(raw: np.ndarray, fmt: int, channels: int, device: Optional[int] = None) -> np.ndarray:
    """Interleaved PCM bytes (uint8 array) -> mono float32 on the GPU (``syg_ingest_pcm``)."""
    import torch
    raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
    fb = channels * _ffi.PCM_BYTES[fmt]
    frames = raw.size // fb
    if frames == 0:
        return np.zeros(0, dtype=np.float32)
    eng = _ffi.engine(device)
    dev = torch.device("cuda", eng.device)
    d_raw = torch.from_numpy(raw[: frames * fb]).to(dev)
    d_out = torch.empty(frames, dtype=torch.float32, device=dev)
    eng.ingest_pcm_dev(d_raw.data_ptr(), fmt, channels, frames, d_out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    return d_out.cpu().numpy()


def pcm_to_planes(raw: np.ndarray, fmt: int, channels: int, device: Optional[int] = None) -> np.ndarray:
    """Interleaved PCM bytes (uint8 array) -> float32 ``(channels, frames)`` on the GPU: one H2D copy of the payload, one
    ``syg_ingest_pcm_channels`` launch, one D2H copy of the planes."""
    import torch
    raw = np.ascontiguousarray(raw).view(np.uint8).reshape(-1)
    fb = channels * _ffi.PCM_BYTES[fmt]
    frames = raw.size // fb
    if frames == 0:
        return np.zeros((channels, 0), dtype=np.float32)
    eng = _ffi.engine(device)
    dev = torch.device("cuda", eng.device)
    pitch = _ffi.plane_pitch(frames)
    d_raw = torch.from_numpy(raw[: frames * fb]).to(dev)
    d_out = torch.empty(channels * pitch, dtype=torch.float32, device=dev)
    eng.ingest_pcm_channels_dev(d_raw.data_ptr(), fmt, channels, frames, d_out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream)
    return d_out.cpu().numpy().reshape(channels, pitch)[:, :frames]
