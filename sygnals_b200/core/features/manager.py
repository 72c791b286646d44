"""Mirror of ``sygnals/core/features/manager.py:78-445`` (``extract_features``) on the B200 engine.

Same signature, feature-name strings, column order (order of ``features``; ``['all']`` = sorted known names), frame count
(``1 + len(y)//hop`` when centred, manager.py:149-157), time axis (``(i*hop + frame_length//2)/sr``, manager.py:166-169),
naming (``mfcc_i``, ``contrast_band_i``, ``contrast_delta``, manager.py:337-343,365-369), the injected
``spectral_centroid`` column when ``spectral_bandwidth`` is requested first (manager.py:296-301), error types and output
formats.  The arithmetic is ONE fused kernel family on the GPU (FP32); columns are widened to float64.  A feature the reference
fails on is logged and left out, the others are returned (manager.py:394-397; ``_ffi.failing_features``), and NaN rows of the
reference (contrast whose band 0 holds bin 0 only) come back as NaN.

Differences, by design: features without a CUDA kernel raise ``NotImplementedError`` instead of running on the CPU, and
only power-of-two ``frame_length`` in [32, 8192] is supported.
"""
from __future__ import annotations

import logging
from typing import Any, Dict, List, Optional

import numpy as np

from ... import _ffi
from ...batch import feature_row_names

logger = logging.getLogger(__name__)

# names the reference knows (manager.py:38-69 with time_domain.py:231-241, frequency_domain.py:392-399)
_FRAME_BASED_FEATURES = ("mean_amplitude", "std_dev_amplitude", "skewness", "kurtosis", "peak_amplitude", "crest_factor",
                         "signal_entropy", "zero_crossing_rate", "rms_energy", "hnr", "jitter", "shimmer")
_SPECTRUM_BASED_FEATURES = ("spectral_centroid", "spectral_bandwidth", "spectral_flatness", "spectral_rolloff",
                            "dominant_frequency")
_SPECTROGRAM_BASED_FEATURES = ("spectral_contrast",)
_MELSPEC_BASED_FEATURES = ("mfcc",)
_ALL_KNOWN_FEATURES = set(_FRAME_BASED_FEATURES) | set(_SPECTRUM_BASED_FEATURES) | set(_SPECTROGRAM_BASED_FEATURES) | set(
    _MELSPEC_BASED_FEATURES)
# names with a CUDA kernel in libsygb200
ENGINE_FEATURES = frozenset(_ffi.FEATURE_IDS)


class FeatureExtractionError(Exception):
    """Custom exception for errors during feature extraction (manager.py:72-74)."""


def frame_times(num_frames: int, sr: int, hop_length: int, frame_length: int, center: bool) -> np.ndarray:
    off = frame_length // 2 if center else 0
    return ((np.arange(num_frames) * hop_length + off) / float(sr)).astype(np.float64)


def extract_features(y, sr: int, features: List[str], frame_length: int = 2048, hop_length: int = 512, center: bool = True,
                     window: str = "hann", feature_params: Optional[Dict[str, Dict[str, Any]]] = None,
                     output_format: str = "dataframe"):
    feature_params = feature_params or {}
    if features == ["all"]:
        features = sorted(_ALL_KNOWN_FEATURES)
    unknown_features = [f for f in features if f not in _ALL_KNOWN_FEATURES]
    if unknown_features:
        raise ValueError(f"Unknown feature(s) requested: {unknown_features}. Available: {sorted(list(_ALL_KNOWN_FEATURES))}")
    y = np.asarray(y)
    if y.ndim != 1:
        raise ValueError("Input audio signal 'y' must be a 1D array.")
    if output_format not in ("dataframe", "dict_of_arrays"):
        raise ValueError(f"Unsupported output format: {output_format}. Choose 'dataframe' or 'dict_of_arrays'.")
    no_kernel = [f for f in features if f not in ENGINE_FEATURES]
    if no_kernel:
        raise NotImplementedError(f"feature(s) {no_kernel} have no CUDA kernel in sygnals_b200 (they stay on the reference path); "
                                  f"available on the engine: {sorted(ENGINE_FEATURES)}")

    def empty():
        if output_format == "dataframe":
            import pandas as pd
            return pd.DataFrame()
        return {"time": np.array([], dtype=np.float64)}

    eng = _ffi.engine()
    num_frames = eng.frame_count(len(y), frame_length, hop_length, center) if frame_length % 2 == 0 else (
        1 + len(y) // hop_length if center else (1 + (len(y) - frame_length) // hop_length if len(y) >= frame_length else 0))
    if num_frames <= 0:
        logger.warning("Signal is too short for the given frame/hop length and centering setting. No frames generated.")
        return empty()
    # order of evaluation = order of the list, duplicates skipped (manager.py:230-232); bandwidth-before-centroid injects
    # the centroid column at that point (manager.py:296-301)
    plan: List[str] = []
    for f in features:
        if f in plan:
            continue
        if f == "spectral_bandwidth" and "spectral_centroid" not in plan:
            plan.append("spectral_centroid")
        plan.append(f)
    # a feature the reference fails on is logged and left out, the others are returned (manager.py:394-397); the rest still run in
    # one engine call
    for f, why in _ffi.failing_features(eng.lib, plan, sr, frame_length, feature_params).items():
        logger.error(f"Error calculating feature '{f}': {why}")
        plan.remove(f)
    times = frame_times(num_frames, sr, hop_length, frame_length, center)
    if not plan:
        logger.warning("No features were successfully extracted or passed final checks.")
        return empty() if output_format == "dataframe" else {"time": times}
    try:
        p = _ffi.reference_params(eng.lib, sr, plan, frame_length, hop_length, center, window, feature_params)
        rows = eng.features_host(y.astype(np.float32, copy=False), eng.units_clips(1, len(y)), p)[0]
    except (ValueError, NotImplementedError):
        raise
    except Exception as e:  # CUDA / allocation failure
        raise FeatureExtractionError(f"Failed to compute features on the B200 engine: {e}") from e
    names = feature_row_names(plan, feature_params)
    final: Dict[str, np.ndarray] = {"time": times}
    for n, r in zip(names, rows):
        final[n] = r.astype(np.float64)
    if output_format == "dataframe":
        import pandas as pd
        try:
            idx = pd.to_timedelta(final.pop("time"), unit="s")
            df = pd.DataFrame(final, index=idx)
            df.index.name = "time"
            return df
        except Exception as e:
            raise FeatureExtractionError(f"Error creating output DataFrame: {e}")
    return final
