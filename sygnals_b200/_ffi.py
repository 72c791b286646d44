"""ctypes binding of ``libsygb200.so`` (C ABI: ``include/sygb200.h``).

The library is the product: hand-written sm_100a CUDA kernels behind plain-C entry points.  There is no CPU
fallback -- if the library is missing, or no CUDA device is present, every call raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libsygb200.so"

SYG_OK = 0
SYG_E_BADARG, SYG_E_SHAPE, SYG_E_CUDA, SYG_E_NOMEM, SYG_E_UNSUPPORTED = -1, -2, -3, -4, -5

FEATURE_IDS = {
    "mfcc": 0,
    "spectral_contrast": 1,
    "spectral_centroid": 2,
    "spectral_rolloff": 3,
    "rms_energy": 4,
    "crest_factor": 5,
    "peak_amplitude": 6,
    "spectral_bandwidth": 7,
    "spectral_flatness": 8,
    "dominant_frequency": 9,
    "mean_amplitude": 10,
    "std_dev_amplitude": 11,
    "zero_crossing_rate": 12,
    "skewness": 13,
    "kurtosis": 14,
    "signal_entropy": 15,
}
WINDOW_IDS = {"hann": 0, "hanning": 0, "hamming": 1, "blackman": 2, "boxcar": 3, "rectangular": 3, "rect": 3, "ones": 3}
PAD_IDS = {"constant": 0, "reflect": 1}
OUT_COMPLEX, OUT_MAGNITUDE, OUT_POWER = 0, 1, 2
SCALING_IDS = {"density": 0, "spectrum": 1}
AGG_IDS = {"mean": 0, "std": 1, "median": 2, "min": 3, "max": 4}      # formatters.py:39-45
PCM_U8, PCM_S16, PCM_S24, PCM_S32, PCM_F32 = 0, 1, 2, 3, 4              # sample formats of a WAV 'data' payload
PCM_BYTES = {PCM_U8: 1, PCM_S16: 2, PCM_S24: 3, PCM_S32: 4, PCM_F32: 4}
MAX_FEATURES = 16
# syg_debug_last_feature_kernel / syg_debug_last_welch_path values (include/sygb200.h)
FK_WARP_WIDE, FK_WARP, FK_SPEC44K, FK_SPEC22K, FK_SPEC44KL, FK_RESIDENT, FK_BLOCK, FK_MIXED = 1, 2, 3, 4, 5, 6, 7, 8
WELCH_WARP, WELCH_BLOCK, WELCH_MIXED = 1, 2, 3


class EngineError(RuntimeError):
    """CUDA / allocation failure inside libsygb200."""


class SygUnits(C.Structure):
    _fields_ = [("n_units", C.c_int64), ("unit_len", C.c_int64), ("unit_stride", C.c_int64), ("total_len", C.c_int64),
                ("unit_starts", C.c_void_p), ("unit_valid", C.c_void_p)]


class SygRaggedUnits(C.Structure):
    """Units of their own lengths: unit u is y[starts[u], starts[u] + lengths[u]) (host int64 tables)."""
    _fields_ = [("n_units", C.c_int64), ("total_len", C.c_int64), ("starts", C.c_void_p), ("lengths", C.c_void_p)]


class SygFeatureParams(C.Structure):
    _fields_ = [("sr", C.c_int32), ("frame_length", C.c_int32), ("hop_length", C.c_int32), ("center", C.c_int32),
                ("window", C.c_int32), ("n_features", C.c_int32), ("features", C.c_int32 * MAX_FEATURES),
                ("n_mels", C.c_int32), ("fmin", C.c_double), ("fmax", C.c_double), ("power", C.c_double),
                ("n_mfcc", C.c_int32), ("dct_type", C.c_int32), ("dct_ortho", C.c_int32), ("lifter", C.c_double),
                ("contrast_n_bands", C.c_int32), ("contrast_fmin", C.c_double), ("contrast_quantile", C.c_double),
                ("roll_percent", C.c_double), ("entropy_bins", C.c_int32)]


def default_library_path() -> str:
    return os.path.join(_HERE, LIB_NAME)


class Library:
    """Loaded libsygb200 with typed prototypes."""

    def __init__(self, path: Optional[str] = None):
        path = path or default_library_path()
        if not os.path.exists(path):
            raise ImportError(
                f"{path} not found: build it with `python -m sygnals_b200.build` (nvcc, sm_100a). "
                "sygnals_b200 has no CPU fallback.")
        self.path = path
        self.dll = C.CDLL(path)
        d = self.dll
        vp, i32, i64, f32, f64, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_size_t
        PU, PP, PR = C.POINTER(SygUnits), C.POINTER(SygFeatureParams), C.POINTER(SygRaggedUnits)
        protos = {
            "syg_version": (C.c_char_p, []),
            "syg_last_error": (C.c_char_p, []),
            "syg_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
            "syg_ctx_destroy": (None, [vp]),
            "syg_ctx_set_workspace_limit": (C.c_int, [vp, sz]),
            "syg_ctx_sm_count": (C.c_int, [vp]),
            "syg_ctx_profile_enable": (C.c_int, [vp, C.c_int]),
            "syg_ctx_profile_read": (C.c_int, [vp, vp, vp, C.c_int]),
            "syg_feature_params_default": (None, [PP]),
            "syg_features_rows": (C.c_int, [PP, C.POINTER(i32)]),
            "syg_frame_count": (i64, [i64, i32, i32, i32]),
            "syg_features_f32": (C.c_int, [vp, vp, PU, PP, vp, vp]),
            "syg_features_host_f32": (C.c_int, [vp, vp, PU, PP, vp]),
            "syg_features_host_pcm16": (C.c_int, [vp, vp, PU, PP, vp]),
            "syg_pcm16_to_f32": (C.c_int, [vp, vp, vp, i64, vp]),
            "syg_ingest_pcm": (C.c_int, [vp, vp, i32, i32, i64, vp, vp]),
            "syg_features_host_pcm": (C.c_int, [vp, vp, i32, i32, PU, PP, vp]),
            "syg_ingest_pcm_channels": (C.c_int, [vp, vp, i32, i32, i64, vp, vp]),
            "syg_psd_welch_host_pcm_channels": (C.c_int, [vp, vp, i32, i32, PU, f64, i32, i32, i32, i32, i32, i32, vp, vp]),
            "syg_segment_vectors_host_pcm_channels": (C.c_int, [vp, vp, i32, i32, PU, PP, vp, vp]),
            "syg_segment_vectors_f32": (C.c_int, [vp, vp, PU, PP, vp, vp, vp]),
            "syg_segment_vectors_host_f32": (C.c_int, [vp, vp, PU, PP, vp, vp]),
            "syg_segment_vectors_host_pcm": (C.c_int, [vp, vp, i32, i32, PU, PP, vp, vp]),
            "syg_ragged_frame_offsets": (i64, [PR, i32, i32, i32, vp]),
            "syg_features_ragged_f32": (C.c_int, [vp, vp, PR, PP, vp, vp]),
            "syg_features_ragged_host_f32": (C.c_int, [vp, vp, PR, PP, vp]),
            "syg_segment_vectors_ragged_f32": (C.c_int, [vp, vp, PR, PP, vp, vp, vp]),
            "syg_segment_vectors_ragged_host_f32": (C.c_int, [vp, vp, PR, PP, vp, vp]),
            "syg_mel_spectrogram_f32": (C.c_int, [vp, vp, PU, PP, i32, vp, vp]),
            "syg_mel_spectrogram_host_f32": (C.c_int, [vp, vp, PU, PP, i32, vp]),
            "syg_mel_spectrogram_ragged_f32": (C.c_int, [vp, vp, PR, PP, i32, vp, vp]),
            "syg_mel_spectrogram_ragged_host_f32": (C.c_int, [vp, vp, PR, PP, i32, vp]),
            "syg_stft_f32": (C.c_int, [vp, vp, PU, i32, i32, i32, i32, i32, i32, i32, vp, vp]),
            "syg_stft_host_f32": (C.c_int, [vp, vp, PU, i32, i32, i32, i32, i32, i32, i32, vp]),
            "syg_psd_welch_f32": (C.c_int, [vp, vp, PU, f64, i32, i32, i32, i32, i32, i32, vp, vp, vp]),
            "syg_psd_welch_host_f32": (C.c_int, [vp, vp, PU, f64, i32, i32, i32, i32, i32, i32, vp, vp]),
            "syg_aggregate_f32": (C.c_int, [vp, vp, i64, i32, i64, vp, vp, i32, vp, vp, vp]),
            "syg_segment_count": (i64, [i64, f64, f64, f64, i32, f64, C.POINTER(i64), C.POINTER(i64)]),
            "syg_segment_table": (i64, [i64, f64, f64, f64, i32, f64, vp, vp, i64]),
            "syg_mfcc_from_logmel_f64": (C.c_int, [vp, vp, i64, i32, i64, i32, i32, i32, f64, vp, vp]),
            "syg_spectral_contrast_from_mag_f32": (C.c_int, [vp, vp, i32, i64, f64, i32, f64, f64, vp, vp]),
            "syg_debug_last_stft_path": (C.c_int, []),
            "syg_debug_last_features_resident": (C.c_int, []),
            "syg_debug_last_feature_frames": (i64, []),
            "syg_debug_last_mel_form": (C.c_int, []),
            "syg_debug_last_feature_kernel": (C.c_int, []),
            "syg_debug_last_finalize": (None, [C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]),
            "syg_debug_last_welch_path": (C.c_int, []),
            "syg_debug_last_mixed_threads": (C.c_int, []),
            "syg_debug_set_resident_min_groups": (None, [C.c_int]),
            "syg_debug_window": (C.c_int, [i32, i32, i32, vp]),
            "syg_debug_mel_basis": (C.c_int, [i32, i32, i32, f64, f64, vp]),
            "syg_debug_dct": (C.c_int, [i32, i32, i32, i32, f64, vp]),
            "syg_debug_contrast_bands": (C.c_int, [i32, i32, i32, f64, f64, vp, vp, vp]),
            "syg_host_alloc": (C.c_int, [C.POINTER(vp), sz]),
            "syg_host_free": (C.c_int, [vp]),
        }
        self.symbols = tuple(protos)
        for name, (res, args) in protos.items():
            fn = getattr(d, name)          # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args

    # ------------------------------------------------------------------ error mapping
    def last_error(self) -> str:
        return (self.dll.syg_last_error() or b"").decode("utf-8", "replace")

    def check(self, rc: int) -> None:
        if rc == SYG_OK:
            return
        msg = self.last_error()
        if rc in (SYG_E_BADARG, SYG_E_SHAPE):
            raise ValueError(msg)
        if rc == SYG_E_UNSUPPORTED:
            raise NotImplementedError(msg)
        if rc == SYG_E_NOMEM:
            raise MemoryError(msg)
        raise EngineError(msg)

    def version(self) -> str:
        return self.dll.syg_version().decode()

    # ------------------------------------------------------------------ host-only helpers (no device needed)
    def frame_count(self, n_samples: int, frame_length: int, hop_length: int, center: bool = True) -> int:
        return int(self.dll.syg_frame_count(int(n_samples), int(frame_length), int(hop_length), int(bool(center))))

    def segment_table(self, total_samples: int, sr: float, segment_length_sec: float, overlap_ratio: float = 0.0,
                      pad: bool = True, min_segment_length_sec: Optional[float] = None):
        """(seg_len, seg_hop, starts[int64], valid[int32]) with segmentation.py:62-114 integer arithmetic."""
        mn = -1.0 if min_segment_length_sec is None else float(min_segment_length_sec)
        seg_len, seg_hop = C.c_int64(0), C.c_int64(0)
        n = self.dll.syg_segment_count(int(total_samples), float(sr), float(segment_length_sec), float(overlap_ratio),
                                       int(bool(pad)), mn, C.byref(seg_len), C.byref(seg_hop))
        if n < 0:
            self.check(int(n))
        starts = np.zeros(int(n), dtype=np.int64)
        valid = np.zeros(int(n), dtype=np.int32)
        if n:
            m = self.dll.syg_segment_table(int(total_samples), float(sr), float(segment_length_sec), float(overlap_ratio),
                                           int(bool(pad)), mn, starts.ctypes.data, valid.ctypes.data, int(n))
            assert m == n
        return int(seg_len.value), int(seg_hop.value), starts, valid

    def ragged_frame_offsets(self, units: SygRaggedUnits, frame_length: int, hop_length: int, center: bool = True) -> np.ndarray:
        """int64 ``[n_units + 1]``: F_0 = 0, F_{u+1} = F_u + T_u (T_u = frame_count(lengths[u], ...))."""
        out = np.zeros(int(units.n_units) + 1, dtype=np.int64)
        n = self.dll.syg_ragged_frame_offsets(C.byref(units), int(frame_length), int(hop_length), int(bool(center)), out.ctypes.data)
        if n < 0:
            self.check(int(n))
        return out

    def last_feature_frames(self) -> int:
        """Frames the feature kernels processed in the last features / segment-vectors call of this process."""
        return int(self.dll.syg_debug_last_feature_frames())

    def last_finalize(self) -> tuple:
        """(frames per tile, CTAs, tiles) of the last finalize launch of a feature call."""
        tt, ctas, tiles = C.c_int32(0), C.c_int64(0), C.c_int64(0)
        self.dll.syg_debug_last_finalize(C.byref(tt), C.byref(ctas), C.byref(tiles))
        return int(tt.value), int(ctas.value), int(tiles.value)

    def debug_window(self, window: int, win_length: int, n_fft: int) -> np.ndarray:
        out = np.zeros(n_fft, dtype=np.float32)
        self.check(self.dll.syg_debug_window(window, win_length, n_fft, out.ctypes.data))
        return out

    def debug_mel_basis(self, sr: int, n_fft: int, n_mels: int, fmin: float = 0.0, fmax: float = 0.0) -> np.ndarray:
        out = np.zeros((n_mels, 1 + n_fft // 2), dtype=np.float32)
        self.check(self.dll.syg_debug_mel_basis(sr, n_fft, n_mels, fmin, fmax, out.ctypes.data))
        return out

    def debug_dct(self, n_mfcc: int, n_mels: int, dct_type: int = 2, ortho: bool = True, lifter: float = 0.0) -> np.ndarray:
        out = np.zeros((n_mfcc, n_mels), dtype=np.float32)
        self.check(self.dll.syg_debug_dct(n_mfcc, n_mels, dct_type, int(ortho), lifter, out.ctypes.data))
        return out

    def debug_contrast_bands(self, sr: int, n_fft: int, n_bands: int = 6, fmin: float = 200.0, quantile: float = 0.02):
        lo = np.zeros(max(n_bands + 1, 0), dtype=np.int32)
        cnt = np.zeros(max(n_bands + 1, 0), dtype=np.int32)
        nq = np.zeros(max(n_bands + 1, 0), dtype=np.int32)
        self.check(self.dll.syg_debug_contrast_bands(sr, n_fft, n_bands, fmin, quantile, lo.ctypes.data, cnt.ctypes.data,
                                                     nq.ctypes.data))
        return lo, cnt, nq

    def default_params(self) -> SygFeatureParams:
        p = SygFeatureParams()
        self.dll.syg_feature_params_default(C.byref(p))
        return p


_lib_lock = threading.Lock()
_lib: Optional[Library] = None


def library() -> Library:
    """The process-wide product library (``sygnals_b200/libsygb200.so``)."""
    global _lib
    with _lib_lock:
        if _lib is None:
            _lib = Library()
        return _lib


def mfcc_count(feature_params: Optional[dict] = None) -> int:
    """MFCC rows of a request: librosa slices the DCT of the n_mels log-mel rows (``dct(S)[:n_mfcc]``), so at most n_mels."""
    m = (feature_params or {}).get("mfcc", {})
    return min(int(m.get("n_mfcc", 13)), int(m.get("n_mels", 128)))


def failing_features(lib: Library, features: Sequence[str], sr: int, frame_length: int, feature_params: Optional[dict] = None) -> dict:
    """{feature: reason} for the requested features whose computation raises in the reference (which then leaves them out):
    * ``spectral_contrast`` when its octave bands cannot be planned: a band edge at or above Nyquist, a band without FFT bins,
      bad ``n_bands`` / ``fmin`` / ``quantile`` (librosa's ParameterError, or the IndexError of an empty band).  The engine's own
      band planner decides; more than 11 bands are left to the engine, which refuses them.
    * ``mfcc`` with a negative lifter, or a positive one and ``n_mfcc > n_mels`` (librosa's lifter has n_mfcc entries, the DCT
      output only n_mels rows, and the product does not broadcast)."""
    fp = feature_params or {}
    out = {}
    if "spectral_contrast" in features:
        c = fp.get("spectral_contrast", {})
        n_bands = int(c.get("n_bands", 6))
        if n_bands <= 11:
            try:
                lib.debug_contrast_bands(int(sr), int(frame_length), n_bands, float(c.get("fmin", 200.0)), float(c.get("quantile", 0.02)))
            except ValueError as e:
                out["spectral_contrast"] = str(e)
    if "mfcc" in features:
        m = fp.get("mfcc", {})
        lifter = float(m.get("lifter", 0.0))
        if lifter < 0:
            out["mfcc"] = f"MFCC lifter={lifter} must be a non-negative number"
        elif lifter > 0 and int(m.get("n_mfcc", 13)) > int(m.get("n_mels", 128)):
            out["mfcc"] = "the lifter has n_mfcc entries but the DCT only n_mels rows: operands could not be broadcast together"
    return out


def make_params(lib: Library, sr: int, features: Sequence[str], frame_length: int = 2048, hop_length: int = 512,
                center: bool = True, window: str = "hann", feature_params: Optional[dict] = None) -> SygFeatureParams:
    """Translate extract_features() arguments (manager.py:78-88) into the C parameter block."""
    fp = feature_params or {}
    p = lib.default_params()
    p.sr = int(sr)
    p.frame_length = int(frame_length)
    p.hop_length = int(hop_length)
    p.center = int(bool(center))
    if not isinstance(window, str) or window.lower() not in WINDOW_IDS:
        raise NotImplementedError(f"window={window!r}: supported windows are {sorted(set(WINDOW_IDS))}")
    p.window = WINDOW_IDS[window.lower()]
    if len(features) > MAX_FEATURES:
        raise NotImplementedError(f"at most {MAX_FEATURES} feature families per call")
    p.n_features = len(features)
    for i, name in enumerate(features):
        if name not in FEATURE_IDS:
            raise NotImplementedError(f"feature {name!r} has no CUDA kernel in sygnals_b200")
        p.features[i] = FEATURE_IDS[name]
    m = fp.get("mfcc", {})
    # manager.py:213-217 reads n_mels/fmin/fmax/power for the mel stage; cepstral.py:24-27 the DCT ones
    p.n_mels = int(m.get("n_mels", 128))
    p.fmin = float(m.get("fmin", 0.0))
    fmax = m.get("fmax", None)
    p.fmax = 0.0 if fmax is None else float(fmax)
    p.power = float(m.get("power", 2.0))
    p.n_mfcc = int(m.get("n_mfcc", 13))
    p.dct_type = int(m.get("dct_type", 2))
    norm = m.get("norm", "ortho")
    if norm not in ("ortho", None):
        raise ValueError(f"norm={norm!r} is not a valid DCT normalisation")
    p.dct_ortho = 1 if norm == "ortho" else 0
    p.lifter = float(m.get("lifter", 0.0))
    c = fp.get("spectral_contrast", {})
    p.contrast_n_bands = int(c.get("n_bands", 6))
    p.contrast_fmin = float(c.get("fmin", 200.0))
    p.contrast_quantile = float(c.get("quantile", 0.02))
    r = fp.get("spectral_rolloff", {})
    p.roll_percent = float(r.get("roll_percent", 0.85))
    p.entropy_bins = int(fp.get("signal_entropy", {}).get("num_bins", 10))
    return p


def reference_params(lib: Library, sr: int, features: Sequence[str], frame_length: int = 2048, hop_length: int = 512,
                     center: bool = True, window: str = "hann", feature_params: Optional[dict] = None) -> SygFeatureParams:
    """:func:`make_params` for the entry points that mirror the reference.  A feature the reference would fail on
    (:func:`failing_features`) raises ValueError (the manager leaves such features out before it gets here), and the parameter block
    asks for :func:`mfcc_count` coefficients, the rows ``batch.feature_row_names`` names.  ``make_params`` itself passes ``n_mfcc``
    through, so the C ABI still rejects more coefficients than mel bands."""
    for name, why in failing_features(lib, features, sr, frame_length, feature_params).items():
        raise ValueError(f"{name}: {why}")
    fp = dict(feature_params or {})
    if "mfcc" in fp:
        fp["mfcc"] = dict(fp["mfcc"], n_mfcc=mfcc_count(fp))
    return make_params(lib, sr, features, frame_length, hop_length, center, window, fp)


def plane_pitch(n_frames: int) -> int:
    """Floats between the planes of ``syg_ingest_pcm_channels``: ``n_frames`` rounded up to a multiple of 4."""
    return (int(n_frames) + 3) // 4 * 4


def _check_out(a, shape, dtype, what: str) -> None:
    """A caller's preallocated result must be exactly what the library writes: the D2H copies trust its size and layout."""
    if not isinstance(a, np.ndarray) or a.dtype != dtype or a.shape != tuple(shape) or not a.flags.c_contiguous or not a.flags.writeable:
        raise ValueError(f"{what} must be a writeable C-contiguous {np.dtype(dtype).name} array of shape {tuple(shape)}")


def _f32c(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


class Engine:
    """One ``syg_ctx`` (device context + plan cache).  Thread-compatible; calls are serialised inside the library."""

    def __init__(self, device: int = 0, lib: Optional[Library] = None):
        self.lib = lib or library()
        h = C.c_void_p()
        self.lib.check(self.lib.dll.syg_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.dll.syg_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self) -> int:
        return int(self.lib.dll.syg_ctx_sm_count(self._h))

    def set_workspace_limit(self, nbytes: int) -> None:
        self.lib.check(self.lib.dll.syg_ctx_set_workspace_limit(self._h, int(nbytes)))

    def profile_enable(self, on: bool = True) -> None:
        self.lib.check(self.lib.dll.syg_ctx_profile_enable(self._h, int(on)))

    def profile_read(self, reset: bool = True) -> dict:
        """{'frame': (ms, launches), 'finalize': (...), 'welch': (...), 'other': (...)} summed since the last reset
        ('other' = ingest + aggregation kernels)."""
        ms = (C.c_double * 4)()
        n = (C.c_int64 * 4)()
        self.lib.check(self.lib.dll.syg_ctx_profile_read(self._h, C.addressof(ms), C.addressof(n), int(reset)))
        return {k: (float(ms[i]), int(n[i])) for i, k in enumerate(("frame", "finalize", "welch", "other"))}

    # ------------------------------------------------------------------ geometry helpers
    @staticmethod
    def units_clips(n_units: int, unit_len: int, total_len: Optional[int] = None, stride: Optional[int] = None) -> SygUnits:
        u = SygUnits()
        u.n_units, u.unit_len = int(n_units), int(unit_len)
        u.unit_stride = int(unit_len if stride is None else stride)
        u.total_len = int(n_units * unit_len if total_len is None else total_len)
        u.unit_starts, u.unit_valid = None, None
        return u

    @staticmethod
    def units_table(starts_ptr: int, valid_ptr: int, n_units: int, unit_len: int, total_len: int) -> SygUnits:
        u = SygUnits()
        u.n_units, u.unit_len, u.unit_stride, u.total_len = int(n_units), int(unit_len), 0, int(total_len)
        u.unit_starts, u.unit_valid = starts_ptr, valid_ptr
        return u

    @staticmethod
    def ragged_units(starts, lengths, total_len: int) -> SygRaggedUnits:
        """Ragged unit tables (host int64 copies; the returned structure keeps them alive)."""
        st = np.ascontiguousarray(starts, dtype=np.int64).reshape(-1)
        ln = np.ascontiguousarray(lengths, dtype=np.int64).reshape(-1)
        if st.shape != ln.shape:
            raise ValueError("starts and lengths must have the same length")
        u = SygRaggedUnits()
        u.n_units, u.total_len = int(st.shape[0]), int(total_len)
        u.starts, u.lengths = (st.ctypes.data, ln.ctypes.data) if st.size else (None, None)
        u._keep = (st, ln)
        return u

    def rows(self, p: SygFeatureParams) -> int:
        n = C.c_int32(0)
        self.lib.check(self.lib.dll.syg_features_rows(C.byref(p), C.byref(n)))
        return int(n.value)

    def frame_count(self, n, fl, hop, center=True) -> int:
        return self.lib.frame_count(n, fl, hop, center)

    # ------------------------------------------------------------------ host-buffer entry points (numpy in/out)
    def features_host(self, y: np.ndarray, units: SygUnits, p: SygFeatureParams, out: Optional[np.ndarray] = None,
                      y_ptr: Optional[int] = None, keep=None) -> np.ndarray:
        """float32 [n_units, n_rows, T] for the units of ``y`` (1-D float32 host buffer, or a raw pointer)."""
        rows = self.rows(p)
        T = self.frame_count(units.unit_len, p.frame_length, p.hop_length, p.center)
        if out is None:
            out = np.empty((units.n_units, rows, T), dtype=np.float32)
        if y_ptr is None and getattr(y, "dtype", None) == np.int16:       # 16-bit PCM: widened on the device (x / 32768)
            y = np.ascontiguousarray(y)
            self.lib.check(self.lib.dll.syg_features_host_pcm16(self._h, y.ctypes.data, C.byref(units), C.byref(p), out.ctypes.data))
            return out
        if y_ptr is None:
            y = _f32c(y)
            y_ptr = y.ctypes.data
        self.lib.check(self.lib.dll.syg_features_host_f32(self._h, y_ptr, C.byref(units), C.byref(p), out.ctypes.data))
        return out

    def features_host_pcm16(self, y_ptr: int, units: SygUnits, p: SygFeatureParams, out: np.ndarray) -> np.ndarray:
        """Raw-pointer form of the PCM16 host path (pinned int16 buffer)."""
        self.lib.check(self.lib.dll.syg_features_host_pcm16(self._h, y_ptr, C.byref(units), C.byref(p), out.ctypes.data))
        return out

    def features_host_pcm(self, raw_ptr: int, fmt: int, channels: int, units: SygUnits, p: SygFeatureParams,
                          out: Optional[np.ndarray] = None) -> np.ndarray:
        """``features_host`` for an interleaved PCM payload in host memory (``units`` count frames of the payload)."""
        rows = self.rows(p)
        T = self.frame_count(units.unit_len, p.frame_length, p.hop_length, p.center)
        if out is None:
            out = np.empty((units.n_units, rows, T), dtype=np.float32)
        self.lib.check(self.lib.dll.syg_features_host_pcm(self._h, raw_ptr, int(fmt), int(channels), C.byref(units), C.byref(p),
                                                          out.ctypes.data))
        return out

    def segment_vectors_host(self, y_ptr: int, units: SygUnits, p: SygFeatureParams, agg_ids: Sequence[int],
                             out: Optional[np.ndarray] = None, fmt: Optional[int] = None, channels: int = 1) -> np.ndarray:
        """float64 ``[n_units, n_rows]``: per-unit features aggregated over the unit's frames on the device (formatters.py:51-163).
        ``fmt=None``: ``y_ptr`` points at float32 mono samples; else at an interleaved PCM payload of format ``fmt``."""
        rows = self.rows(p)
        if len(agg_ids) != rows:
            raise ValueError("one aggregation id per feature row")
        if out is None:
            out = np.empty((units.n_units, rows), dtype=np.float64)
        agg = (C.c_int32 * max(1, rows))(*[int(a) for a in agg_ids])
        if fmt is None:
            rc = self.lib.dll.syg_segment_vectors_host_f32(self._h, y_ptr, C.byref(units), C.byref(p), C.addressof(agg), out.ctypes.data)
        else:
            rc = self.lib.dll.syg_segment_vectors_host_pcm(self._h, y_ptr, int(fmt), int(channels), C.byref(units), C.byref(p),
                                                           C.addressof(agg), out.ctypes.data)
        self.lib.check(rc)
        return out

    def segment_vectors_dev(self, y_ptr: int, units: SygUnits, p: SygFeatureParams, agg_ids: Sequence[int], out_ptr: int,
                            stream: int = 0) -> None:
        """Device form: float32 samples in HBM -> float64 ``[n_units, n_rows]`` in HBM, asynchronous on ``stream``."""
        agg = (C.c_int32 * max(1, len(agg_ids)))(*[int(a) for a in agg_ids])
        self.lib.check(self.lib.dll.syg_segment_vectors_f32(self._h, y_ptr, C.byref(units), C.byref(p), C.addressof(agg), out_ptr,
                                                            stream or None))

    def mfcc_from_logmel_dev(self, S_ptr: int, n_units: int, n_mels: int, T: int, n_mfcc: int, dct_type: int, ortho: bool, lifter: float,
                             out_ptr: int, stream: int = 0) -> None:
        self.lib.check(self.lib.dll.syg_mfcc_from_logmel_f64(self._h, S_ptr, int(n_units), int(n_mels), int(T), int(n_mfcc), int(dct_type),
                                                             int(bool(ortho)), float(lifter), out_ptr, stream or None))

    def spectral_contrast_from_mag_dev(self, S_ptr: int, n_bins: int, T: int, sr: float, n_bands: int, fmin: float, quantile: float,
                                       out_ptr: int, stream: int = 0) -> None:
        self.lib.check(self.lib.dll.syg_spectral_contrast_from_mag_f32(self._h, S_ptr, int(n_bins), int(T), float(sr), int(n_bands),
                                                                       float(fmin), float(quantile), out_ptr, stream or None))

    def ingest_pcm_dev(self, raw_ptr: int, fmt: int, channels: int, n_frames: int, out_ptr: int, stream: int = 0) -> None:
        """Interleaved PCM in HBM -> mono float32 in HBM (load_audio(mono=True) arithmetic)."""
        self.lib.check(self.lib.dll.syg_ingest_pcm(self._h, raw_ptr, int(fmt), int(channels), int(n_frames), out_ptr, stream or None))

    def ingest_pcm_channels_dev(self, raw_ptr: int, fmt: int, channels: int, n_frames: int, out_ptr: int, stream: int = 0) -> None:
        """Interleaved PCM in HBM -> float32 planes ``out[c * plane_pitch(n_frames) + i]`` in HBM (load_audio(mono=False))."""
        self.lib.check(self.lib.dll.syg_ingest_pcm_channels(self._h, raw_ptr, int(fmt), int(channels), int(n_frames), out_ptr,
                                                            stream or None))

    def psd_welch_host_pcm_channels(self, raw_ptr: int, fmt: int, channels: int, units: SygUnits, fs: float, window: int, nperseg: int,
                                    noverlap: int, nfft: int, detrend: bool = True, scaling: int = 0, stats: bool = False,
                                    out: Optional[tuple] = None):
        """Welch PSD per (unit, channel) of an interleaved PCM payload in host memory (``units`` count frames): psd
        ``[n_units, channels, 1 + nfft/2]`` float32 and, with ``stats``, ``[n_units, channels, 3]`` (rms, crest, peak).  ``out``:
        optional preallocated (psd, stats) arrays of those shapes (e.g. ``pinned_empty``)."""
        nfft_eff = nfft if nfft and nfft > 0 else nperseg
        n, ch = int(units.n_units), int(channels)
        if out is None:
            out = (np.empty((n, ch, nfft_eff // 2 + 1), dtype=np.float32), np.empty((n, ch, 3), dtype=np.float32) if stats else None)
        psd, st = out
        _check_out(psd, (n, ch, nfft_eff // 2 + 1), np.float32, "out[0]")
        if stats:
            _check_out(st, (n, ch, 3), np.float32, "out[1]")
        else:
            st = None
        self.lib.check(self.lib.dll.syg_psd_welch_host_pcm_channels(
            self._h, raw_ptr, int(fmt), ch, C.byref(units), float(fs), int(window), int(nperseg), int(noverlap), int(nfft_eff),
            int(bool(detrend)), int(scaling), psd.ctypes.data, st.ctypes.data if st is not None else None))
        return (psd, st) if stats else psd

    def segment_vectors_host_pcm_channels(self, raw_ptr: int, fmt: int, channels: int, units: SygUnits, p: SygFeatureParams,
                                          agg_ids: Sequence[int], out: Optional[np.ndarray] = None) -> np.ndarray:
        """float64 ``[n_units, channels, n_rows]``: ``segment_vectors_host`` per channel of an interleaved PCM payload, no mix-down."""
        rows = self.rows(p)
        if len(agg_ids) != rows:
            raise ValueError("one aggregation id per feature row")
        if out is None:
            out = np.empty((int(units.n_units), int(channels), rows), dtype=np.float64)
        _check_out(out, (int(units.n_units), int(channels), rows), np.float64, "out")
        agg = (C.c_int32 * max(1, rows))(*[int(a) for a in agg_ids])
        self.lib.check(self.lib.dll.syg_segment_vectors_host_pcm_channels(self._h, raw_ptr, int(fmt), int(channels), C.byref(units),
                                                                          C.byref(p), C.addressof(agg), out.ctypes.data))
        return out

    def stft_host(self, y: np.ndarray, units: SygUnits, n_fft: int, hop: int, win_length: int, window: int = 0,
                  center: bool = True, pad_mode: int = 0, out_kind: int = OUT_COMPLEX, out: Optional[np.ndarray] = None) -> np.ndarray:
        """``out``: optional preallocated result (e.g. ``pinned_empty``: the D2H copies then run at PCIe speed)."""
        y = _f32c(y)
        T = self.frame_count(units.unit_len, n_fft, hop, center)
        B = 1 + n_fft // 2
        dt = np.complex64 if out_kind == OUT_COMPLEX else np.float32
        if out is None:
            out = np.empty((units.n_units, B, T), dtype=dt)
        elif out.dtype != dt or out.shape != (units.n_units, B, T) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous array of shape (n_units, 1 + n_fft/2, T) and the output dtype")
        self.lib.check(self.lib.dll.syg_stft_host_f32(self._h, y.ctypes.data, C.byref(units), int(n_fft), int(hop),
                                                      int(win_length), int(window), int(bool(center)), int(pad_mode),
                                                      int(out_kind), out.ctypes.data))
        return out

    def psd_welch_host(self, y: np.ndarray, units: SygUnits, fs: float, window: int, nperseg: int, noverlap: int,
                       nfft: int, detrend: bool = True, scaling: int = 0, stats: bool = False):
        y = _f32c(y)
        nfft_eff = nfft if nfft and nfft > 0 else nperseg
        psd = np.empty((units.n_units, nfft_eff // 2 + 1), dtype=np.float32)
        st = np.empty((units.n_units, 3), dtype=np.float32) if stats else None
        self.lib.check(self.lib.dll.syg_psd_welch_host_f32(
            self._h, y.ctypes.data, C.byref(units), float(fs), int(window), int(nperseg), int(noverlap), int(nfft_eff),
            int(bool(detrend)), int(scaling), psd.ctypes.data, st.ctypes.data if stats else None))
        return (psd, st) if stats else psd

    def features_ragged_host(self, y: np.ndarray, units: SygRaggedUnits, p: SygFeatureParams, out: Optional[np.ndarray] = None) -> np.ndarray:
        """float32 ``[n_rows, F]`` for ragged units of the 1-D float32 host buffer ``y`` (row r of frame t of unit u at column F_u + t)."""
        y = _f32c(y)
        F = int(self.lib.ragged_frame_offsets(units, p.frame_length, p.hop_length, p.center)[-1])
        if out is None:
            out = np.empty((self.rows(p), F), dtype=np.float32)
        self.lib.check(self.lib.dll.syg_features_ragged_host_f32(self._h, y.ctypes.data, C.byref(units), C.byref(p), out.ctypes.data))
        return out

    def segment_vectors_ragged_host(self, y: np.ndarray, units: SygRaggedUnits, p: SygFeatureParams, agg_ids: Sequence[int],
                                    out: Optional[np.ndarray] = None) -> np.ndarray:
        """float64 ``[n_units, n_rows]``: each ragged unit's frames aggregated per row (a unit without frames gives a NaN row)."""
        rows = self.rows(p)
        if len(agg_ids) != rows:
            raise ValueError("one aggregation id per feature row")
        y = _f32c(y)
        if out is None:
            out = np.empty((int(units.n_units), rows), dtype=np.float64)
        agg = (C.c_int32 * max(1, rows))(*[int(a) for a in agg_ids])
        self.lib.check(self.lib.dll.syg_segment_vectors_ragged_host_f32(self._h, y.ctypes.data, C.byref(units), C.byref(p),
                                                                        C.addressof(agg), out.ctypes.data))
        return out

    def mel_spectrogram_host(self, y: np.ndarray, units: SygUnits, p: SygFeatureParams, db: bool = True,
                             out: Optional[np.ndarray] = None) -> np.ndarray:
        """float32 ``[n_units, n_mels, T]``: S_db (``db``) or S_mel of the units of ``y`` (1-D float32 host buffer); ``p`` without
        features (``n_features = 0``)."""
        y = _f32c(y)
        T = self.frame_count(units.unit_len, p.frame_length, p.hop_length, p.center)
        if out is None:
            out = np.empty((int(units.n_units), max(int(p.n_mels), 0), T), dtype=np.float32)
        self.lib.check(self.lib.dll.syg_mel_spectrogram_host_f32(self._h, y.ctypes.data, C.byref(units), C.byref(p), int(bool(db)),
                                                                 out.ctypes.data))
        return out

    def mel_spectrogram_ragged_host(self, y: np.ndarray, units: SygRaggedUnits, p: SygFeatureParams, db: bool = True,
                                    out: Optional[np.ndarray] = None) -> np.ndarray:
        """float32 ``[n_mels, F]`` for ragged units of the 1-D float32 host buffer ``y`` (band m of frame t of unit u at column
        F_u + t)."""
        y = _f32c(y)
        F = int(self.lib.ragged_frame_offsets(units, p.frame_length, p.hop_length, p.center)[-1])
        if out is None:
            out = np.empty((max(int(p.n_mels), 0), F), dtype=np.float32)
        self.lib.check(self.lib.dll.syg_mel_spectrogram_ragged_host_f32(self._h, y.ctypes.data, C.byref(units), C.byref(p),
                                                                        int(bool(db)), out.ctypes.data))
        return out

    # ------------------------------------------------------------------ device-pointer entry points (async)
    def mel_spectrogram_dev(self, y_ptr: int, units: SygUnits, p: SygFeatureParams, db: bool, out_ptr: int, stream: int = 0) -> None:
        """Device form of ``mel_spectrogram_host``: float32 ``[n_units, n_mels, T]`` in HBM, asynchronous on ``stream``."""
        self.lib.check(self.lib.dll.syg_mel_spectrogram_f32(self._h, y_ptr, C.byref(units), C.byref(p), int(bool(db)), out_ptr,
                                                            stream or None))

    def mel_spectrogram_ragged_dev(self, y_ptr: int, units: SygRaggedUnits, p: SygFeatureParams, db: bool, out_ptr: int,
                                   stream: int = 0) -> None:
        """Device form of ``mel_spectrogram_ragged_host``: float32 ``[n_mels, F]`` in HBM, asynchronous on ``stream``."""
        self.lib.check(self.lib.dll.syg_mel_spectrogram_ragged_f32(self._h, y_ptr, C.byref(units), C.byref(p), int(bool(db)), out_ptr,
                                                                   stream or None))

    def features_dev(self, y_ptr: int, units: SygUnits, p: SygFeatureParams, out_ptr: int, stream: int = 0) -> None:
        self.lib.check(self.lib.dll.syg_features_f32(self._h, y_ptr, C.byref(units), C.byref(p), out_ptr, stream or None))

    def features_ragged_dev(self, y_ptr: int, units: SygRaggedUnits, p: SygFeatureParams, out_ptr: int, stream: int = 0) -> None:
        """Device form of ``features_ragged_host``: float32 ``[n_rows, F]`` in HBM, asynchronous on ``stream``."""
        self.lib.check(self.lib.dll.syg_features_ragged_f32(self._h, y_ptr, C.byref(units), C.byref(p), out_ptr, stream or None))

    def segment_vectors_ragged_dev(self, y_ptr: int, units: SygRaggedUnits, p: SygFeatureParams, agg_ids: Sequence[int], out_ptr: int,
                                   stream: int = 0) -> None:
        """Device form of ``segment_vectors_ragged_host``: float64 ``[n_units, n_rows]`` in HBM, asynchronous on ``stream``."""
        agg = (C.c_int32 * max(1, len(agg_ids)))(*[int(a) for a in agg_ids])
        self.lib.check(self.lib.dll.syg_segment_vectors_ragged_f32(self._h, y_ptr, C.byref(units), C.byref(p), C.addressof(agg), out_ptr,
                                                                   stream or None))

    def stft_dev(self, y_ptr: int, units: SygUnits, n_fft: int, hop: int, win_length: int, window: int, center: bool,
                 pad_mode: int, out_kind: int, out_ptr: int, stream: int = 0) -> None:
        self.lib.check(self.lib.dll.syg_stft_f32(self._h, y_ptr, C.byref(units), int(n_fft), int(hop), int(win_length),
                                                 int(window), int(bool(center)), int(pad_mode), int(out_kind), out_ptr,
                                                 stream or None))

    def psd_welch_dev(self, y_ptr: int, units: SygUnits, fs: float, window: int, nperseg: int, noverlap: int, nfft: int,
                      detrend: bool, scaling: int, psd_ptr: int, stats_ptr: int = 0, stream: int = 0) -> None:
        self.lib.check(self.lib.dll.syg_psd_welch_f32(self._h, y_ptr, C.byref(units), float(fs), int(window), int(nperseg),
                                                      int(noverlap), int(nfft), int(bool(detrend)), int(scaling), psd_ptr,
                                                      stats_ptr or None, stream or None))

    def aggregate_dev(self, feats_ptr: int, n_seg: int, n_rows: int, row_stride: int, agg_ids: Sequence[int], out_ptr: int,
                      seg_off_ptr: int = 0, seg_len_ptr: int = 0, fixed_len: int = 0, stream: int = 0) -> None:
        """format_feature_vectors_per_segment on device buffers (float32 in, float64 [n_seg, n_rows] out)."""
        agg = (C.c_int32 * max(1, n_rows))(*[int(a) for a in agg_ids])
        self.lib.check(self.lib.dll.syg_aggregate_f32(self._h, feats_ptr, int(n_seg), int(n_rows), int(row_stride), seg_off_ptr or None,
                                                      seg_len_ptr or None, int(fixed_len), C.addressof(agg), out_ptr, stream or None))

    # ------------------------------------------------------------------ pinned host memory
    def pinned_empty(self, shape, dtype=np.float32) -> np.ndarray:
        """numpy array backed by cudaHostAlloc memory; the block is released when the array (and every view of it) is collected."""
        import weakref
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        n = count * dtype.itemsize
        p = C.c_void_p()
        self.lib.check(self.lib.dll.syg_host_alloc(C.byref(p), max(n, 1)))
        buf = (C.c_char * max(n, 1)).from_address(p.value)
        # views keep `buf` alive through .base; when the last one dies the finalizer frees the page-locked block
        weakref.finalize(buf, self.lib.dll.syg_host_free, C.c_void_p(p.value))
        return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)


_engines: dict = {}
_engine_lock = threading.Lock()


def engine(device: Optional[int] = None) -> Engine:
    """Cached per-device Engine of the product library."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if os.environ.get("SYGB200_DEVICE") is None else int(
            os.environ["SYGB200_DEVICE"])
    with _engine_lock:
        e = _engines.get(device)
        if e is None:
            e = Engine(device)
            _engines[device] = e
        return e


def shutdown() -> None:
    with _engine_lock:
        for e in _engines.values():
            e.close()
        _engines.clear()
