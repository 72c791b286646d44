"""Requests the reference handles in a degenerate way, through the package's public entry points, against the float64 oracle.

The reference's ``extract_features`` (manager.py:374-397, restated in oracle/sygnals_oracle.py) leaves out a feature whose
computation raises and returns the others, and returns whatever rows librosa produced, NaN included.  The cases:

* ``spectral_contrast`` whose octave bands cannot be planned (a band edge at or above Nyquist, e.g. the default bands at 8 kHz;
  a band without FFT bins, e.g. 44.1 kHz at frame_length 32): the reference drops contrast and returns the other features.
* contrast whose band 0 ``[0, fmin]`` holds bin 0 only (bin spacing above fmin): librosa averages an empty slice for that band and
  power_to_db's top_db clamp spreads the NaN, so every contrast row is NaN on every frame.
* ``mfcc`` with ``n_mfcc > n_mels``: librosa slices the DCT output, n_mels rows come back; with a lifter as well the lifter does
  not broadcast and MFCC is dropped.

Result dicts are compared whole: keys in order (with the centroid column that spectral_bandwidth injects), frame times, the NaN
pattern of every row, and the values at the tolerances of tests/test_parity_cabi.py.  The additive batch entry points
(extract_features_batch, extract_features_ragged, clip_vectors, channel_vectors) have no per-feature fallback: they RAISE
ValueError where the manager drops a feature, so a caller never gets a row layout other than the one it asked for; NaN contrast
rows and truncated MFCCs they return like the manager.

A request the engine does not serve must raise NotImplementedError (the plugin then hands it to the reference), and only the
documented refusals in REFUSALS may do so.  Each failing sweep case is printed as a literal for the regression table.
"""
import re

import numpy as np
import pytest

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi, batch
from sygnals_b200.core.features import manager
from sygnals_b200.utils import synth
from test_parity_cabi import check_rows, row_tol

ALL = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor", "peak_amplitude",
       "spectral_bandwidth", "spectral_flatness", "dominant_frequency", "mean_amplitude", "std_dev_amplitude", "zero_crossing_rate",
       "skewness", "kurtosis", "signal_entropy"]


def req(sr, fl, hop, feats, fp=None, center=True, window="hann", L=None, seed=0):
    return dict(sr=sr, fl=fl, hop=hop, feats=list(feats), fp=fp or {}, center=center, window=window, L=4 * fl if L is None else L,
                seed=seed)


# Each of these failed before the manager dropped unplannable contrast, the plan wrote NaN for a single-bin band 0 and
# the mirror layers asked for min(n_mfcc, n_mels) coefficients.
REGRESSIONS = [
    req(8000, 512, 128, ["spectral_contrast", "rms_energy"]),                              # default bands past Nyquist at 8 kHz
    req(11025, 1024, 256, ["mfcc", "spectral_contrast", "spectral_centroid"]),             # ... and at 11.025 kHz
    req(44100, 32, 8, ["spectral_contrast", "rms_energy"]),                                # a band without FFT bins
    req(44100, 128, 32, ["spectral_contrast", "rms_energy"]),                              # band 0 = bin 0 only: all contrast NaN
    req(48000, 128, 32, ["rms_energy", "spectral_contrast", "zero_crossing_rate"]),
    req(16000, 64, 16, ["spectral_contrast"]),
    req(22050, 64, 16, ["spectral_bandwidth", "spectral_contrast"]),
    req(16000, 512, 128, ["mfcc", "rms_energy"], {"mfcc": {"n_mfcc": 20, "n_mels": 10}}),  # n_mfcc > n_mels: n_mels rows
    req(16000, 512, 128, ["rms_energy", "mfcc", "spectral_centroid"], {"mfcc": {"n_mfcc": 20, "n_mels": 10, "lifter": 22.0}}),  # dropped
]


def _largest_prime(n):
    m, p, big = n, 2, 1
    while p * p <= m:
        while m % p == 0:
            m //= p
            big = p
        p += 1
    return max(big, m) if m > 1 else big


def _mfcc(r):
    return r["fp"].get("mfcc", {})


# (what, does the request fall under it, message): the only NotImplementedErrors a request may meet
REFUSALS = [
    ("n_mels > 256", lambda r: "mfcc" in r["feats"] and int(_mfcc(r).get("n_mels", 128)) > 256,
     r"n_mels=\d+: supported range is \[1, 256\]|n_mfcc=\d+: supported range is \[1, 256\]"),
    ("entropy bins outside [1, 16]", lambda r: "signal_entropy" in r["feats"]
     and not 1 <= int(r["fp"].get("signal_entropy", {}).get("num_bins", 10)) <= 16,
     r"signal_entropy num_bins=-?\d+: supported range is \[1, 16\]"),
    ("prime factors above 13", lambda r: r["fl"] & (r["fl"] - 1) != 0 and _largest_prime(r["fl"] // 2 if r["fl"] % 2 == 0 else r["fl"]) > 13,
     r"frame_length=\d+: only lengths whose prime factors are at most 13 are supported"),
    ("plan exceeds shared memory", lambda r: "mfcc" in r["feats"] and r["fl"] == 2048 and int(_mfcc(r).get("n_mels", 128)) <= 2,
     r"the plan needs \d+ bytes of shared memory per block, the device allows \d+"),
]

REFUSAL_CASES = [
    req(22050, 1024, 256, ["mfcc"], {"mfcc": {"n_mels": 300}}),
    req(22050, 1024, 256, ["rms_energy", "mfcc"], {"mfcc": {"n_mels": 300, "n_mfcc": 300}}),
    req(16000, 512, 128, ["signal_entropy"], {"signal_entropy": {"num_bins": 0}}),
    req(16000, 512, 128, ["rms_energy", "signal_entropy"], {"signal_entropy": {"num_bins": 17}}),
    req(16000, 544, 136, ["rms_energy"]),                                                  # 544 = 2^5 * 17
    req(16000, 2048, 512, ["mfcc"], {"mfcc": {"n_mels": 1, "n_mfcc": 1}}),
    req(96000, 2048, 512, ["mfcc", "rms_energy"], {"mfcc": {"n_mels": 2}}),
]


@pytest.fixture(params=BACKENDS)
def eng(request, monkeypatch):
    e = get_engine(request.param)
    monkeypatch.setattr(_ffi, "engine", lambda device=None: e)
    return e


def signal(r, n=None, seed=0):
    """four partials across the band over white noise (well defined for clips of a few samples too)"""
    n = r["L"] if n is None else n
    rng = np.random.default_rng(1000 * r["seed"] + seed)
    t = np.arange(n) / r["sr"]
    y = 0.05 * rng.standard_normal(n)
    for f, a, ph in zip(rng.uniform(30.0, 0.45 * r["sr"], 4), rng.uniform(0.1, 0.5, 4), rng.uniform(0, 2 * np.pi, 4)):
        y += a * np.sin(2 * np.pi * f * t + ph)
    y = y.astype(np.float32)
    if r["seed"] % 3 == 1:
        y[: len(y) // 3] = 0.0                                   # silence: the FP32 noise floor paths
    return y


def kw(r):
    return dict(frame_length=r["fl"], hop_length=r["hop"], center=r["center"], window=r["window"], feature_params=r["fp"])


def oracle(r, y):
    return orc.extract_features(np.asarray(y, dtype=np.float64), r["sr"], list(r["feats"]), **kw(r))


def contrast_ok(r, y):
    """frames without bins below the FP32 noise floor (the mask of test_edge_clips_vs_oracle)"""
    if len(y) == 0 or (not r["center"] and len(y) < r["fl"]):
        return None
    S = np.abs(orc.compute_stft(np.asarray(y, dtype=np.float64), n_fft=r["fl"], hop_length=r["hop"], window=r["window"],
                                center=r["center"]))
    return S.min(axis=0) >= 1e-5 * S.max(axis=0)


def refusal(r, e):
    for what, applies, pattern in REFUSALS:
        if applies(r) and re.search(pattern, str(e)):
            return what
    return None


def compare_rows(r, names, got, ref, ok):
    """got / ref: {name: [T]}; NaN patterns equal, the rows without NaN within the parity tolerances"""
    if len(ref["time"]) == 0:                                    # no frames: the reference returns the time axis only
        assert all(len(got[n]) == 0 for n in names)
        return
    for n in names:
        assert np.array_equal(np.isnan(got[n]), np.isnan(ref[n])), f"{n}: NaN pattern {np.isnan(got[n]).sum()} vs {np.isnan(ref[n]).sum()}"
    fin = [n for n in names if not np.isnan(ref[n]).any()]
    if fin and len(ref[fin[0]]):
        check_rows(fin, np.stack([got[n] for n in fin]), np.stack([ref[n] for n in fin]), bin_hz=r["sr"] / r["fl"], nyq=r["sr"] / 2,
                   contrast_ok=ok)


def check_manager(r):
    """manager.extract_features in both output formats against the oracle; 'refused: ...' / 'ok'"""
    y = signal(r)
    ref = oracle(r, y)
    try:
        got = manager.extract_features(y, r["sr"], r["feats"], output_format="dict_of_arrays", **kw(r))
    except NotImplementedError as e:
        what = refusal(r, e)
        assert what is not None, f"undocumented refusal: {e}"
        return f"refused: {what}"
    assert list(got) == list(ref)
    assert len(got["time"]) == len(ref["time"])
    np.testing.assert_allclose(got["time"], ref["time"], rtol=0, atol=1e-9)
    names = [k for k in ref if k != "time"]
    compare_rows(r, names, got, ref, contrast_ok(r, y))
    df = manager.extract_features(y, r["sr"], r["feats"], output_format="dataframe", **kw(r))
    if not names or not len(ref["time"]):
        assert df.empty
    else:
        assert list(df.columns) == names and len(df) == len(ref["time"])
        for n in names:
            np.testing.assert_array_equal(df[n].to_numpy(), got[n])
    return "ok"


def expects_drop(r):
    return _ffi.failing_features(_ffi.engine().lib, r["feats"], r["sr"], r["fl"], r["fp"])


def check_batch(r):
    """extract_features_batch, extract_features_ragged, clip_vectors: names, NaN patterns, values per clip"""
    sr, fl = r["sr"], r["fl"]
    L0 = r["L"]
    L1 = max(1, L0 // 2 + 7)
    clips = [signal(r, L0), signal(r, L1, seed=1)]
    dropped = expects_drop(r)
    calls = [lambda: batch.extract_features_batch(np.stack([clips[0], signal(r, L0, seed=2)]), sr, r["feats"], **kw(r)),
             lambda: batch.extract_features_ragged(clips, sr, r["feats"], **kw(r)),
             lambda: batch.clip_vectors(clips, sr, r["feats"], aggregation="mean", **kw(r))]
    if dropped:
        for c in calls:                                          # the additive APIs raise where the manager drops
            with pytest.raises(ValueError):
                c()
        return "raised"
    try:
        names, out = calls[0]()
    except NotImplementedError as e:
        assert refusal(r, e) is not None, f"undocumented refusal: {e}"
        return "refused"
    assert names == batch.feature_row_names(r["feats"], r["fp"])
    assert out.shape[:2] == (2, len(names))
    for c, y in enumerate([clips[0], signal(r, L0, seed=2)]):
        ref = oracle(r, y)
        assert out.shape[2] == len(ref["time"])
        compare_rows(r, names, dict(zip(names, out[c])), ref, contrast_ok(r, y))
    rag = calls[1]()
    assert rag["names"] == names
    foff = rag["frame_offsets"]
    if len(names) > 64:                                          # the aggregation kernel's documented limit
        with pytest.raises(NotImplementedError, match="aggregation supports at most 64 rows per call"):
            calls[2]()
        vec = None
    else:
        vnames, vec = calls[2]()
        assert vnames == names and vec.shape == (2, len(names))
    for c, y in enumerate(clips):
        ref = oracle(r, y)
        part = rag["features"][:, foff[c]:foff[c + 1]]
        assert part.shape[1] == len(ref["time"])
        compare_rows(r, names, dict(zip(names, part)), ref, contrast_ok(r, y))
        for i, n in enumerate(names if vec is not None else []):                            # formatters.py:31-36: all-NaN (or no frames) -> NaN
            want = orc.AGGREGATION_FUNCS["mean"](ref[n]) if len(ref["time"]) else np.nan
            if np.isnan(want):
                assert np.isnan(vec[c, i]), f"clip {c} {n}: {vec[c, i]} where the reference aggregates to NaN"
            else:
                assert abs(vec[c, i] - want) <= 2 * np.max(row_tol(n, [want], bin_hz=sr / fl, nyq=sr / 2) if n != "zero_crossing_rate"
                                                           else 1e-6), f"clip {c} {n}: {vec[c, i]} vs {want}"
    return "ok"


# ------------------------------------------------------------------------------------------------ the seeded sweep
SRS = [8000, 11025, 16000, 22050, 32000, 44100, 48000, 96000]
FLS = [32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 400, 441, 1000]


def sweep_case(i):
    rng = np.random.default_rng(7000 + i)
    sr = int(rng.choice(SRS))
    fl = int(rng.choice(FLS))
    hop = int(rng.choice([fl // 4, fl // 2, fl, fl + 1, 2 * fl, max(1, fl // 3) + 1]))
    center = bool(rng.random() < 0.6)
    window = str(rng.choice(["hann", "hamming", "blackman", "boxcar"]))
    if rng.random() < 0.2:
        L = int(rng.integers(1, fl))                             # shorter than one frame
    else:
        L = int(fl + rng.integers(0, min(24 * hop, 6 * fl)))
    core = list(rng.choice(["mfcc", "spectral_contrast"], size=int(rng.integers(1, 3)), replace=False))
    rest = [f for f in ALL if f not in core]
    feats = [str(f) for f in core + list(rng.choice(rest, size=int(rng.integers(0, 4)), replace=False))]
    rng.shuffle(feats)                                           # a dropped feature between kept ones
    fp = {}
    if "spectral_contrast" in feats:
        fp["spectral_contrast"] = {"n_bands": int(rng.integers(1, 12)), "fmin": float(rng.choice([50.0, 200.0, 1000.0, 4000.0])),
                                   "quantile": float(rng.choice([0.01, 0.02, 0.5, 0.99]))}
    if "mfcc" in feats:
        n_mels = int(rng.choice([1, 2, 3, 8, 10, 20, 40, 64, 128, 256]))
        m = {"n_mels": n_mels, "n_mfcc": int(rng.choice([max(1, n_mels - 3), n_mels, n_mels + 1, n_mels + 12]))}
        kind = rng.integers(0, 4)
        if kind == 1:
            m["fmin"], m["fmax"] = 0.4 * sr, 0.1 * sr            # fmin > fmax
        elif kind == 2:
            m["fmax"] = 0.75 * sr                                # fmax > sr / 2
        if rng.random() < 0.2:
            m["lifter"] = 22.0
        fp["mfcc"] = m
    if "signal_entropy" in feats:
        fp["signal_entropy"] = {"num_bins": int(rng.integers(1, 17))}
    if "spectral_rolloff" in feats:
        fp["spectral_rolloff"] = {"roll_percent": float(rng.choice([0.85, 0.5, 0.99]))}
    return req(sr, fl, hop, feats, fp, center=center, window=window, L=L, seed=i)


N_SWEEP, N_CHUNK = 96, 12
SWEEP = [sweep_case(i) for i in range(N_SWEEP)]


def _run_table(table, fn):
    failed = []
    for r in table:
        try:
            fn(r)
        except AssertionError as e:
            failed.append(f"    req({r['sr']}, {r['fl']}, {r['hop']}, {r['feats']!r}, {r['fp']!r}, center={r['center']}, "
                          f"window={r['window']!r}, L={r['L']}, seed={r['seed']}),  # {str(e).splitlines()[0][:160]}")
    assert not failed, "failing requests (paste into REGRESSIONS):\n" + "\n".join(failed)


# ------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("k", range(len(REGRESSIONS)))
def test_named_regressions_through_the_manager(eng, k):
    assert check_manager(REGRESSIONS[k]) == "ok"


@pytest.mark.parametrize("k", range(len(REGRESSIONS)))
def test_named_regressions_through_the_batch_apis(eng, k):
    assert check_batch(REGRESSIONS[k]) in ("ok", "raised")


def test_named_regressions_are_degenerate():
    """The table stays what its comments say: the oracle drops / NaNs / truncates on each entry."""
    drops = nans = trunc = 0
    for r in REGRESSIONS:
        ref = oracle(r, signal(r))
        names = batch.feature_row_names(r["feats"], r["fp"])
        drops += any(n not in ref for n in names if not n.startswith("mfcc_"))
        nans += any(np.isnan(ref[n]).all() for n in ref if n.startswith("contrast_"))
        trunc += "mfcc" in r["feats"] and sum(n.startswith("mfcc_") for n in ref) not in (0, int(_mfcc(r).get("n_mfcc", 13)))
    assert drops >= 3 and nans >= 4 and trunc >= 1


@pytest.mark.parametrize("chunk", range(N_SWEEP // N_CHUNK))
def test_sweep_through_the_manager(eng, chunk):
    _run_table(SWEEP[chunk * N_CHUNK:(chunk + 1) * N_CHUNK], check_manager)


@pytest.mark.parametrize("chunk", range(N_SWEEP // N_CHUNK // 4))
def test_sweep_through_the_batch_apis(eng, chunk):
    """a quarter of the sweep (every fourth case) through the additive batch entry points"""
    _run_table(SWEEP[chunk * 4 * N_CHUNK:(chunk + 1) * 4 * N_CHUNK:4], check_batch)


def test_sweep_covers_the_degenerate_domain():
    """the seeds reach every corner the sweep claims"""
    seen = set()
    for r in SWEEP:
        y = signal(r)
        ref = oracle(r, y)
        m = _mfcc(r)
        if "spectral_contrast" in r["feats"]:
            seen.add("contrast dropped" if "contrast_delta" not in ref else
                     ("contrast NaN" if len(ref["time"]) and np.isnan(ref["contrast_delta"]).all() else "contrast kept"))
        if "mfcc" in r["feats"]:
            n_mfcc, n_mels = int(m.get("n_mfcc", 13)), int(m.get("n_mels", 128))
            seen.add("n_mfcc " + ("<" if n_mfcc < n_mels else ("=" if n_mfcc == n_mels else ">")) + " n_mels")
            seen.add("fmin > fmax" if m.get("fmin", 0) > m.get("fmax", r["sr"]) else ("fmax > sr/2" if m.get("fmax", 0) > r["sr"] / 2 else "mel"))
        seen.add(("short" if r["L"] < r["fl"] else "long") + (" centred" if r["center"] else " uncentred"))
        if r["hop"] > r["fl"]:
            seen.add("hop > frame_length")
        kept = [f for f in r["feats"] if any(k == f or k.startswith(f[:4]) for k in ref)]
        if len(kept) >= 2 and len(kept) < len(r["feats"]):
            seen.add("dropped among kept")
    want = {"contrast dropped", "contrast NaN", "contrast kept", "n_mfcc < n_mels", "n_mfcc = n_mels", "n_mfcc > n_mels", "fmin > fmax",
            "fmax > sr/2", "short centred", "short uncentred", "long centred", "long uncentred", "hop > frame_length", "dropped among kept"}
    assert want <= seen, want - seen


@pytest.mark.parametrize("k", range(len(REFUSAL_CASES)))
def test_documented_refusals(eng, k):
    """each raises NotImplementedError with its documented message, through the manager and the batch API"""
    r = REFUSAL_CASES[k]
    y = signal(r)
    for call in (lambda: manager.extract_features(y, r["sr"], r["feats"], output_format="dict_of_arrays", **kw(r)),
                 lambda: batch.extract_features_batch(y[None], r["sr"], r["feats"], **kw(r))):
        with pytest.raises(NotImplementedError) as ei:
            call()
        assert refusal(r, ei.value) is not None, str(ei.value)


def test_c_abi_keeps_refusing_unplannable_contrast(eng):
    """Only the layers that mirror the reference drop: the C ABI still answers SYG_E_BADARG (ValueError) for bands it cannot plan."""
    for sr, fl in [(8000, 512), (44100, 32)]:
        p = _ffi.make_params(eng.lib, sr, ["rms_energy"], fl, fl // 4)     # reference_params refuses such a request
        p.n_features = 2
        p.features[1] = _ffi.FEATURE_IDS["spectral_contrast"]
        with pytest.raises(ValueError, match="Nyquist|without FFT bins"):
            eng.features_host(np.zeros(4 * fl, np.float32), eng.units_clips(1, 4 * fl), p)


def test_mfcc_row_counts_agree(eng):
    """syg_features_rows, feature_row_names and the manager's columns for n_mfcc below, at and above n_mels"""
    for n_mfcc, n_mels in [(5, 10), (10, 10), (20, 10), (13, 1)]:
        fp = {"mfcc": {"n_mfcc": n_mfcc, "n_mels": n_mels}}
        feats = ["rms_energy", "mfcc", "spectral_centroid"]
        p = _ffi.reference_params(eng.lib, 16000, feats, 512, 128, feature_params=fp)
        names = batch.feature_row_names(feats, fp)
        assert eng.rows(p) == len(names) == 2 + min(n_mfcc, n_mels)
        if n_mfcc > n_mels:                                      # the C ABI itself keeps rejecting the raw request
            raw = _ffi.make_params(eng.lib, 16000, feats, 512, 128, feature_params=fp)
            assert raw.n_mfcc == n_mfcc
            with pytest.raises(ValueError, match=r"n_mfcc must be in \[1, n_mels\]"):
                eng.features_host(np.zeros(2048, np.float32), eng.units_clips(1, 2048), raw)
        got = manager.extract_features(signal(req(16000, 512, 128, feats, fp)), 16000, feats, frame_length=512, hop_length=128,
                                       feature_params=fp, output_format="dict_of_arrays")
        assert [k for k in got if k != "time"] == names


def test_plugin_mixed_request_drops_like_the_reference(eng):
    """The plugin's split of a mixed request (engine features + reference-only ones): a contrast the reference drops is left out
    between kept columns, MFCCs are truncated to n_mels, and the engine columns equal the oracle's."""
    from sygnals_b200 import plugin as plg

    def fake_ref(y, sr, features, **kw):                         # jitter has no kernel; a stand-in for the reference
        return {"time": orc.extract_features(np.asarray(y, np.float64), sr, ["rms_energy"], frame_length=kw["frame_length"],
                                             hop_length=kw["hop_length"])["time"], **{f: np.full(1, 7.0) for f in features}}

    r = req(8000, 512, 128, ["jitter", "spectral_contrast", "rms_energy", "mfcc"], {"mfcc": {"n_mfcc": 20, "n_mels": 10}})
    y = signal(r)
    fn = plg.SygnalsB200Plugin().make_extract_features(original=fake_ref)
    got = fn(y, r["sr"], r["feats"], frame_length=r["fl"], hop_length=r["hop"], feature_params=r["fp"], output_format="dict_of_arrays")
    ref = orc.extract_features(y.astype(np.float64), r["sr"], ["spectral_contrast", "rms_energy", "mfcc"], frame_length=r["fl"],
                               hop_length=r["hop"], feature_params=r["fp"])
    assert list(got) == ["time", "jitter", "rms_energy"] + [f"mfcc_{i}" for i in range(10)]
    assert [k for k in ref if k != "time"] == list(got)[2:]
    compare_rows(r, list(got)[2:], got, ref, None)


def test_vectors_of_units_without_frames(eng):
    """Uncentred clips / segments shorter than a frame have no frames; their vectors are NaN (formatters.py:31-36), also when no unit
    of the call has a frame (the aggregation launch then does not run and the output used to be left unwritten)."""
    sr, fl, hop = 16000, 512, 128
    feats = ["rms_energy", "mfcc"]
    y = signal(req(sr, fl, hop, feats, L=2000))
    for clips in ([y[:300], y[300:700]], [y[:300], y[300:1500]]):
        names, vec = batch.clip_vectors(clips, sr, feats, frame_length=fl, hop_length=hop, center=False)
        assert np.isnan(vec[0]).all() and np.isnan(vec[1]).all() == (len(clips[1]) < fl)
    pcm = np.stack([y, y[::-1]], axis=1).astype(np.float32)
    _, cv = batch.channel_vectors(batch.Payload(pcm.tobytes(), _ffi.PCM_F32, 2, sr), 0.02, feats, frame_length=fl, hop_length=hop,
                                  center=False)                  # 320-sample segments
    assert cv.shape == (7, 2, len(names)) and np.isnan(cv).all()


def test_nan_contrast_on_every_entry_point(eng):
    """band 0 = bin 0 (44.1 kHz, frame_length 128): NaN on the uniform, ragged, segment and PCM-channel launches; the other rows
    finite and equal to the same request without contrast"""
    sr, fl, hop = 44100, 128, 32
    feats = ["rms_energy", "spectral_contrast", "spectral_centroid"]
    y = synth.mixture(6000, sr, seed=3).astype(np.float32)
    names, out = batch.extract_features_batch(np.stack([y[:3000], y[3000:]]), sr, feats, frame_length=fl, hop_length=hop)
    ci = [i for i, n in enumerate(names) if n.startswith("contrast_")]
    oi = [i for i, n in enumerate(names) if not n.startswith("contrast_")]
    assert len(ci) == 7 and np.isnan(out[:, ci]).all() and np.isfinite(out[:, oi]).all()
    _, plain = batch.extract_features_batch(np.stack([y[:3000], y[3000:]]), sr, ["rms_energy", "spectral_centroid"], frame_length=fl,
                                            hop_length=hop)
    np.testing.assert_array_equal(out[:, oi], plain)
    rag = batch.extract_features_ragged([y[:1000], y[1000:4500], y[4500:4600]], sr, feats, frame_length=fl, hop_length=hop)
    assert np.isnan(rag["features"][ci]).all() and np.isfinite(rag["features"][oi]).all()
    seg = batch.segment_features(y, sr, 0.05, feats, frame_length=fl, hop_length=hop)
    assert np.isnan(seg["features"][:, ci]).all() and np.isfinite(seg["features"][:, oi]).all()
    _, vec = batch.clip_vectors([y[:1000], y[1000:4500]], sr, feats, aggregation="max", frame_length=fl, hop_length=hop)
    assert np.isnan(vec[:, ci]).all() and np.isfinite(vec[:, oi]).all()
    pcm = np.stack([y, -0.5 * y], axis=1).astype(np.float32)       # two interleaved channels
    _, cv = batch.channel_vectors(batch.Payload(pcm.tobytes(), _ffi.PCM_F32, 2, sr), 0.05, feats, frame_length=fl, hop_length=hop)
    assert cv.shape[1:] == (2, len(names))
    assert np.isnan(cv[..., ci]).all() and np.isfinite(cv[..., oi]).all()
