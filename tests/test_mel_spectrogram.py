"""Mel and log-mel spectrograms of clips, segments and ragged batches (syg_mel_spectrogram_*, batch.mel_spectrogram_*).

The output is the matrix extract_features builds for its MFCCs (manager.py:213-223): ``S_mel`` (db=False) or
``power_to_db(S_mel, ref=np.max)`` (db=True), per unit, frequency-major.  It is held to the float64 oracle's mel stage
(``oracle_mel``: the calls of extract_features' get_mag / get_logmel, pinned to the oracle's MFCC rows below) on mixtures, to the FP32 yardstick allowance of test_noise_floor.py on tonal / DC /
impulse clips, to exact invariants of power_to_db, to the MFCC rows of the fused feature path, and bit for bit across the host,
device, uniform, segment-table and ragged forms and across workspace chunkings.
"""
import contextlib
import ctypes

import numpy as np
import pytest
import scipy.fftpack

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi, batch
from sygnals_b200.utils import synth
from test_noise_floor import C, K_SPREAD, Yardstick, oracle_on

G31 = 1 << 31
DB_TOL = 1e-3


@pytest.fixture(params=BACKENDS)
def eng(request, monkeypatch):
    e = get_engine(request.param)
    monkeypatch.setattr(_ffi, "engine", lambda device=None: e)        # the batch functions run on this backend
    return e


def on_gpu(eng):
    return eng.test_backend == "gpu"


def kernel(eng):
    return eng.lib.dll.syg_debug_last_feature_kernel()


@contextlib.contextmanager
def workspace_limit(eng, nbytes):
    eng.set_workspace_limit(nbytes)
    try:
        yield
    finally:
        eng.set_workspace_limit(1 << 30)


# name -> (sr, frame_length, hop, n_mels, options, feature kernels that may serve the request).  At n_fft 2048 an MFCC-only plan with
# the interval-form mel runs the Spec44k instantiation (its layout leaves the feature set open); mel power 1 takes the generic kernel.
GEOMS = {
    "cfg1": (22050, 2048, 512, 128, {}, {_ffi.FK_SPEC44K}),
    "cfg3": (16000, 512, 160, 40, {}, {_ffi.FK_WARP}),
    "cfg4": (44100, 2048, 512, 128, {}, {_ffi.FK_SPEC44K}),
    "power1_2048": (44100, 2048, 512, 128, {"power": 1.0}, {_ffi.FK_WARP_WIDE, _ffi.FK_WARP}),
    "mixed400": (16000, 400, 160, 40, {}, {_ffi.FK_MIXED}),
    "block4096": (44100, 4096, 1024, 128, {}, {_ffi.FK_BLOCK}),
    "power1": (22050, 1024, 256, 64, {"power": 1.0}, {_ffi.FK_WARP}),
    "band": (22050, 1024, 256, 64, {"fmin": 50.0, "fmax": 8000.0}, {_ffi.FK_WARP}),
    "hamming": (16000, 512, 160, 40, {"window": "hamming"}, {_ffi.FK_WARP}),
    "nocenter": (16000, 512, 160, 40, {"center": False}, {_ffi.FK_WARP}),
    "mels30": (22050, 512, 128, 30, {}, {_ffi.FK_WARP}),                 # n_mels % 4 != 0: the scalar loads of mel_store
}
EDGES = ("zeros", "dc", "impulse")


def opts(o):
    return dict(center=o.get("center", True), window=o.get("window", "hann"), fmin=o.get("fmin", 0.0), fmax=o.get("fmax"),
                power=o.get("power", 2.0))


def oracle_mel(y, sr, frame_length=2048, hop_length=512, center=True, window="hann", n_mels=128, fmin=0.0, fmax=None, power=2.0,
               db=True):
    """float64 [n_mels, T]: the calls of the oracle's extract_features get_mag (manager.py:184-198) and get_logmel (:213-223) on y,
    through the oracle's librosa (so test_noise_floor.oracle_on can swap the transform).  ``db``: power_to_db(S_mel, ref=np.max)
    (:223), else S_mel (:219-222); ``fmax=None`` is sr / 2 (:216)."""
    L = orc.librosa
    D = L.stft(y=np.asarray(y, dtype=np.float64), n_fft=frame_length, hop_length=hop_length, win_length=frame_length, window=window,
               center=center)
    S = np.abs(D).astype(np.float64)
    S_mel = L.feature.melspectrogram(S=S ** power, sr=sr, n_mels=n_mels, fmin=fmin, fmax=sr / 2.0 if fmax is None else fmax,
                                     n_fft=frame_length)
    return L.power_to_db(S_mel, ref=np.max).astype(np.float64) if db else S_mel


def reference(y, sr, fl, hop, n_mels, o, db):
    o = opts(o)
    return oracle_mel(y, sr, fl, hop, o["center"], o["window"], n_mels, o["fmin"], o["fmax"], o["power"], db)


@pytest.mark.parametrize("o", [{}, {"power": 1.0, "fmin": 50.0, "fmax": 8000.0}, {"window": "hamming", "center": False}])
def test_oracle_mel_is_what_the_oracle_mfcc_transforms(o):
    """oracle_mel(db=True) is the log-mel extract_features hands to mfcc(S=...): its DCT equals the oracle's MFCC rows"""
    sr, fl, hop, n_mels = 22050, 1024, 256, 64
    y = synth.mixture(3 * fl + 77, sr, seed=5).astype(np.float64)
    M = reference(y, sr, fl, hop, n_mels, o, True)
    fp = {"mfcc": {"n_mels": n_mels, "n_mfcc": 20, **{k: v for k, v in o.items() if k in ("power", "fmin", "fmax")}}}
    ref = orc.extract_features(y, sr, ["mfcc"], fl, hop, center=opts(o)["center"], window=opts(o)["window"], feature_params=fp)
    want = np.stack([ref[f"mfcc_{i}"] for i in range(20)])
    got = scipy.fftpack.dct(M, type=2, norm="ortho", axis=0)[:20]
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-9 * max(1.0, np.abs(want).max())


def unit_signals(L, sr):
    """mixtures at two levels (-80 dB clamp), then silence, DC and an impulse; L is not a multiple of any hop used here"""
    return {"mix_a": synth.mixture(L, sr, seed=L), "mix_b": (synth.mixture(L, sr, seed=L + 1) * np.float32(0.01)).astype(np.float32),
            "zeros": synth.edge_clip("zeros", L, sr), "dc": synth.edge_clip("dc", L, sr), "impulse": synth.edge_clip("impulse", L, sr)}


def yardstick_spread(y, sr, fl, hop, n_mels, o, db, gain=1.0):
    """largest deviation of the oracle's mel (+ dB) stage applied to the two FP32 yardstick spectra of y (Hann window)"""
    ref = reference(y, sr, fl, hop, n_mels, o, db)
    spread = np.zeros_like(ref)
    for i in range(2):
        def spectrum(x, n, h, wl, c, pm):
            ys = Yardstick(x, n, h, wl, c, pm)
            return ys.X64 + gain * (ys.Ys[i] - ys.X64)
        with oracle_on(spectrum):
            spread = np.maximum(spread, np.abs(reference(y, sr, fl, hop, n_mels, o, db) - ref))
    return spread


def tolerance(ref, db):
    """S_db: 1e-3 dB; S_mel: 1e-4 S + 1e-6 max S over the unit"""
    return np.full_like(ref, DB_TOL) if db else 1e-4 * np.abs(ref) + 1e-6 * np.abs(ref).max()


def check_db_invariants(got, silent, what):
    assert (got >= np.float32(-80.0)).all(), f"{what}: below -top_db"
    if silent:
        assert (got == 0.0).all(), f"{what}: silence is not 0 dB everywhere"
    else:
        assert got.max() == 0.0, f"{what}: the unit's maximum is {got.max()!r}, not 0 dB"


# ------------------------------------------------------------------------------------------------ 1, 2. parity and invariants
@pytest.mark.parametrize("db", [True, False], ids=["db", "power"])
@pytest.mark.parametrize("geom", list(GEOMS))
def test_parity_with_oracle(eng, geom, db):
    sr, fl, hop, n_mels, o, fks = GEOMS[geom]
    L = 2 * fl + 3 * hop + 7
    sig = unit_signals(L, sr)
    names = list(sig)
    y = np.stack([sig[n] for n in names])
    out = batch.mel_spectrogram_batch(y, sr, fl, hop, n_mels=n_mels, db=db, **opts(o))
    assert kernel(eng) in fks, f"ran feature kernel {kernel(eng)}"
    assert eng.lib.dll.syg_debug_last_features_resident() == 0
    T = eng.frame_count(L, fl, hop, opts(o)["center"])
    assert isinstance(out, np.ndarray) and out.dtype == np.float32 and out.shape == (len(names), n_mels, T)
    for u, n in enumerate(names):
        got = out[u].astype(np.float64)
        ref = reference(y[u], sr, fl, hop, n_mels, o, db)
        tol = tolerance(ref, db)
        if n in EDGES and n != "zeros":
            if opts(o)["window"] != "hann":
                continue                                              # the yardstick spectra are Hann-windowed
            spread = yardstick_spread(y[u], sr, fl, hop, n_mels, o, db)
            spread_c = yardstick_spread(y[u], sr, fl, hop, n_mels, o, db, gain=C)
            tol = tol + np.maximum(K_SPREAD * spread, spread_c)
        d = np.abs(got - ref)
        assert (d <= tol).all(), f"{n}: band/frame {np.unravel_index(np.argmax(d - tol), d.shape)} off by {d.max():.3g}"
        if db:
            check_db_invariants(out[u], n == "zeros", n)
        elif n == "zeros":
            assert (out[u] == 0.0).all()


@pytest.mark.parametrize("db", [True, False], ids=["db", "power"])
@pytest.mark.parametrize("geom", ["cfg3", "cfg4", "mixed400"])
def test_short_and_ragged_clips_match_oracle(eng, geom, db):
    """clips shorter than n_fft and of lengths that are not multiples of the hop, each framed on its own in one ragged call"""
    sr, fl, hop, n_mels, o, fks = GEOMS[geom]
    lengths = [fl // 2 + 3, fl - 1, fl + hop // 2 + 1, 3 * fl + 5]
    clips = [synth.mixture(n, sr, seed=n) for n in lengths]
    r = batch.mel_spectrogram_ragged(clips, sr, fl, hop, n_mels=n_mels, db=db, **opts(o))
    assert kernel(eng) in fks
    mel, foff = r["mel"], r["frame_offsets"]
    assert mel.shape == (n_mels, foff[-1])
    for u, c in enumerate(clips):
        got = mel[:, foff[u]:foff[u + 1]].astype(np.float64)
        ref = reference(c, sr, fl, hop, n_mels, o, db)
        assert got.shape == ref.shape
        assert (np.abs(got - ref) <= tolerance(ref, db)).all(), f"clip {u} ({lengths[u]} samples)"
        if db:
            check_db_invariants(mel[:, foff[u]:foff[u + 1]], False, f"clip {u}")


# ------------------------------------------------------------------------------------------------ 3. the dB the DCT sees
@pytest.mark.parametrize("geom", ["cfg3", "cfg4", "mixed400"])
def test_log_mel_is_what_the_mfcc_path_transforms(eng, geom):
    sr, fl, hop, n_mels, o, _ = GEOMS[geom]
    y = synth.clip_batch(8, 2 * fl + 5 * hop + 3, sr, seed=fl)
    mel_db = batch.mel_spectrogram_batch(y, sr, fl, hop, n_mels=n_mels)
    names, feats = batch.extract_features_batch(y, sr, ["mfcc"], fl, hop, feature_params={"mfcc": {"n_mels": n_mels}})
    assert len(names) == 13
    for u in range(len(y)):
        S = mel_db[u].astype(np.float64)
        if on_gpu(eng):
            from sygnals_b200.core.features import cepstral
            m = cepstral.mfcc(S=S, n_mfcc=13)
        else:
            m = scipy.fftpack.dct(S, type=2, norm="ortho", axis=0)[:13]
        assert np.abs(m - feats[u]).max() <= 1e-4, f"unit {u}"


# ------------------------------------------------------------------------------------------------ 4. paths are bit-identical
def dev_call(eng, fn, y, out_shape):
    """run a device-pointer entry point fn(y_ptr, out_ptr, stream) on y: numpy buffers on the emulator, CUDA tensors on the GPU"""
    if not on_gpu(eng):
        out = np.full(out_shape, np.nan, dtype=np.float32)
        fn(np.ascontiguousarray(y, dtype=np.float32).ctypes.data, out.ctypes.data, 0)
        return out
    import torch
    yd = torch.from_numpy(np.ascontiguousarray(y, dtype=np.float32)).cuda()
    out = torch.full(out_shape, float("nan"), dtype=torch.float32, device="cuda")
    fn(yd.data_ptr(), out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return out.cpu().numpy()


PATH_GEOMS = {"cfg3": (16000, 512, 160, 40), "cfg4": (44100, 2048, 512, 128), "mels30": (22050, 512, 128, 30)}


@pytest.mark.parametrize("db", [True, False], ids=["db", "power"])
@pytest.mark.parametrize("geom", list(PATH_GEOMS))
def test_paths_are_bit_identical(eng, geom, db):
    sr, fl, hop, n_mels = PATH_GEOMS[geom]
    y = synth.long_signal(int(4.3 * sr), sr, seed=fl, block_sec=0.5)
    kw = dict(n_mels=n_mels, db=db, frame_length=fl, hop_length=hop)
    seg = batch.segment_mel_spectrogram(y, sr, 1.0, overlap_ratio=0.5, **kw)
    A, starts, valid, seg_len = seg["mel"], seg["starts"], seg["valid"], seg["seg_len"]
    n = len(starts)
    assert valid[-1] < seg_len                                        # a zero-padded tail segment
    # an explicit segment table (min_segment_length_sec keeps the table path): the same segments
    tab = batch.segment_mel_spectrogram(y, sr, 1.0, overlap_ratio=0.5, min_segment_length_sec=0.05, **kw)
    assert np.array_equal(tab["starts"], starts)
    assert np.array_equal(tab["mel"], A)
    # the segments as clips, zero padded as segment_fixed_length pads them
    clips = np.zeros((n, seg_len), dtype=np.float32)
    for i in range(n):
        clips[i, :valid[i]] = y[starts[i]:starts[i] + valid[i]]
    assert np.array_equal(batch.mel_spectrogram_batch(clips, sr, **kw), A)
    # the full segments as windows of the recording (ragged units), without a copy
    full = np.flatnonzero(valid == seg_len)
    r = batch.mel_spectrogram_ragged(batch.Windows(y, starts[full], valid[full]), sr, **kw)
    for j, i in enumerate(full):
        assert np.array_equal(r["mel"][:, r["frame_offsets"][j]:r["frame_offsets"][j + 1]], A[i]), f"segment {i}"
    # device forms
    p = batch._mel_params(eng.lib, sr, fl, hop, True, "hann", n_mels, 0.0, None, 2.0)
    units = eng.units_clips(n, seg_len, total_len=len(y), stride=seg["seg_hop"])
    D = dev_call(eng, lambda yp, op, st: eng.mel_spectrogram_dev(yp, units, p, db, op, st), y, A.shape)
    assert np.array_equal(D, A)
    ru = eng.ragged_units(starts[full], valid[full], len(y))
    R = dev_call(eng, lambda yp, op, st: eng.mel_spectrogram_ragged_dev(yp, ru, p, db, op, st), y, r["mel"].shape)
    assert np.array_equal(R, r["mel"])
    if on_gpu(eng):
        import torch
        yd = torch.from_numpy(y).cuda()
        out = batch.segment_mel_spectrogram(yd, sr, 1.0, overlap_ratio=0.5, **kw)["mel"]
        assert isinstance(out, torch.Tensor) and out.is_cuda
        assert np.array_equal(out.cpu().numpy(), A)
        out = batch.mel_spectrogram_ragged(batch.Windows(yd, starts[full], valid[full]), sr, **kw)["mel"]
        assert np.array_equal(out.cpu().numpy(), r["mel"])


@pytest.mark.parametrize("db", [True, False], ids=["db", "power"])
def test_workspace_chunks_are_bit_identical(eng, db):
    """a 1 MiB workspace holds 20 units of 101 frames x 128 mels: 60 segments run in several chunks on every form"""
    sr, fl, hop, n_mels = 16000, 512, 160, 128
    y = synth.long_signal(int(6.5 * sr), sr, seed=77, block_sec=0.5)
    kw = dict(n_mels=n_mels, db=db, frame_length=fl, hop_length=hop)
    seg_len, seg_hop, starts, valid = eng.lib.segment_table(len(y), sr, 1.0, 0.9, True)
    assert len(starts) * 101 * n_mels * 4 > 2 * (1 << 20)
    lengths = np.maximum(valid, 1).astype(np.int64)
    p = batch._mel_params(eng.lib, sr, fl, hop, True, "hann", n_mels, 0.0, None, 2.0)
    units = eng.units_clips(len(starts), seg_len, total_len=len(y), stride=seg_hop)
    ru = eng.ragged_units(starts, lengths, len(y))

    def run_all():
        a = batch.segment_mel_spectrogram(y, sr, 1.0, overlap_ratio=0.9, **kw)["mel"]
        b = dev_call(eng, lambda yp, op, st: eng.mel_spectrogram_dev(yp, units, p, db, op, st), y, a.shape)
        c = batch.mel_spectrogram_ragged(batch.Windows(y, starts, lengths), sr, **kw)["mel"]
        d = dev_call(eng, lambda yp, op, st: eng.mel_spectrogram_ragged_dev(yp, ru, p, db, op, st), y, c.shape)
        return a, b, c, d

    ref = run_all()
    with workspace_limit(eng, 1 << 20):
        small = run_all()
    assert np.array_equal(ref[0], ref[1]) and np.array_equal(ref[2], ref[3])
    for r, s in zip(ref, small):
        assert np.array_equal(r, s)


# ------------------------------------------------------------------------------------------------ 5. never the resident epilogue
def test_resident_epilogue_is_never_taken(eng):
    sr, fl, hop, n_mels, o, _ = GEOMS["cfg3"]
    y = synth.clip_batch(6, 16000, sr, seed=9, edges=False)
    eng.lib.dll.syg_debug_set_resident_min_groups(1)
    try:
        batch.extract_features_batch(y, sr, ["mfcc"], fl, hop, feature_params={"mfcc": {"n_mels": n_mels}})
        assert eng.lib.dll.syg_debug_last_features_resident() == 1      # the request is eligible for it
        out = batch.mel_spectrogram_batch(y, sr, fl, hop, n_mels=n_mels)
        assert eng.lib.dll.syg_debug_last_features_resident() == 0
    finally:
        eng.lib.dll.syg_debug_set_resident_min_groups(-1)
    assert kernel(eng) == _ffi.FK_WARP
    for u in range(len(y)):
        ref = reference(y[u], sr, fl, hop, n_mels, o, True)
        assert np.abs(out[u] - ref).max() <= DB_TOL, f"unit {u}"


# ------------------------------------------------------------------------------------------------ 6. refusals and errors
@pytest.mark.parametrize("kw,match", [({"n_mels": 300}, "n_mels=300"), ({"frame_length": 17 * 32, "hop_length": 128}, "prime factors"),
                                      ({"window": "kaiser"}, "window")])
def test_unserved_requests_raise_not_implemented(eng, kw, match):
    y = synth.clip_batch(2, 4000, 16000, seed=1)
    with pytest.raises(NotImplementedError, match=match):
        batch.mel_spectrogram_batch(y, 16000, **kw)
    with pytest.raises(NotImplementedError, match=match):
        batch.mel_spectrogram_ragged(list(y), 16000, **kw)
    with pytest.raises(NotImplementedError, match=match):
        batch.segment_mel_spectrogram(y[0], 16000, 0.1, **kw)


@pytest.mark.parametrize("kw", [{"hop_length": 0}, {"n_mels": 0}, {"power": 0.0}, {"power": -1.0}, {"fmin": 200.0, "fmax": 100.0},
                                {"fmin": 9000.0}])
def test_bad_arguments_raise_value_error(eng, kw):
    y = synth.clip_batch(2, 4000, 16000, seed=1)
    with pytest.raises(ValueError):
        batch.mel_spectrogram_batch(y, 16000, **kw)
    with pytest.raises(ValueError):
        batch.mel_spectrogram_ragged(list(y), 16000, **kw)


def test_c_abi_arguments(eng):
    y = synth.clip_batch(2, 4000, 16000, seed=1).ravel()
    out = np.full(64, 7.0, dtype=np.float32)
    p = batch._mel_params(eng.lib, 16000, 512, 160, True, "hann", 40, 0.0, None, 2.0)
    units = eng.units_clips(2, 4000)
    ru = eng.ragged_units([0, 4000], [4000, 4000], len(y))
    d = eng.lib.dll
    calls = [lambda q, db: d.syg_mel_spectrogram_host_f32(eng._h, y.ctypes.data, ctypes.byref(units), ctypes.byref(q), db, out.ctypes.data),
             lambda q, db: d.syg_mel_spectrogram_f32(eng._h, y.ctypes.data, ctypes.byref(units), ctypes.byref(q), db, out.ctypes.data, None),
             lambda q, db: d.syg_mel_spectrogram_ragged_host_f32(eng._h, y.ctypes.data, ctypes.byref(ru), ctypes.byref(q), db,
                                                                 out.ctypes.data),
             lambda q, db: d.syg_mel_spectrogram_ragged_f32(eng._h, y.ctypes.data, ctypes.byref(ru), ctypes.byref(q), db, out.ctypes.data,
                                                            None)]
    with_features = _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160, feature_params={"mfcc": {"n_mels": 40}})
    for call in calls:
        assert call(with_features, 1) == _ffi.SYG_E_BADARG
        assert "n_features" in eng.lib.last_error()
        assert call(p, 2) == _ffi.SYG_E_BADARG and "db=2" in eng.lib.last_error()
        assert call(p, -1) == _ffi.SYG_E_BADARG
    assert (out == 7.0).all()
    assert d.syg_mel_spectrogram_host_f32(None, y.ctypes.data, ctypes.byref(units), ctypes.byref(p), 1, out.ctypes.data) == _ffi.SYG_E_BADARG
    # no units: nothing written, no failure
    none = eng.units_clips(0, 4000, total_len=len(y))
    assert d.syg_mel_spectrogram_host_f32(eng._h, y.ctypes.data, ctypes.byref(none), ctypes.byref(p), 1, out.ctypes.data) == 0
    assert d.syg_mel_spectrogram_f32(eng._h, y.ctypes.data, ctypes.byref(none), ctypes.byref(p), 0, out.ctypes.data, None) == 0
    assert (out == 7.0).all()


def test_units_without_frames_write_nothing(eng):
    sr, fl, hop = 16000, 512, 160
    y = synth.clip_batch(3, 300, sr, seed=2)
    out = batch.mel_spectrogram_batch(y, sr, fl, hop, n_mels=40, center=False)          # 300 < n_fft: T = 0
    assert out.shape == (3, 40, 0)
    assert batch.mel_spectrogram_batch(np.zeros((0, 4000), np.float32), sr, fl, hop, n_mels=40).shape == (0, 40, 26)
    r = batch.mel_spectrogram_ragged([y[0], y[1]], sr, fl, hop, n_mels=40, center=False)
    assert r["mel"].shape == (40, 0) and list(r["frame_offsets"]) == [0, 0, 0]
    assert batch.mel_spectrogram_ragged([], sr, fl, hop, n_mels=40)["mel"].shape == (40, 0)
    # a unit without frames between two with frames: the columns are the other two units', bit for bit
    a, b = synth.mixture(3000, sr, seed=3), synth.mixture(2500, sr, seed=4)
    r = batch.mel_spectrogram_ragged([a, y[0], b], sr, fl, hop, n_mels=40, center=False)
    foff = r["frame_offsets"]
    assert foff[1] == foff[2]
    assert np.array_equal(r["mel"][:, :foff[1]], batch.mel_spectrogram_batch(a[None], sr, fl, hop, n_mels=40, center=False)[0])
    assert np.array_equal(r["mel"][:, foff[2]:], batch.mel_spectrogram_batch(b[None], sr, fl, hop, n_mels=40, center=False)[0])


# ------------------------------------------------------------------------------------------------ 7. outputs past 2^31 elements
@pytest.mark.gpu
def test_output_past_2g():
    """mel_spectrogram_dev with n_units x n_mels x T > 2^31 (overlapping units of one recording, several workspace chunks): the last
    units sit past element 2^31 and equal, bit for bit, the same units computed on their own; the first ones as well."""
    import torch
    from test_large_offsets import last_units_equal, long_input, need_device_bytes
    eng = get_engine("gpu")
    sr, fl, hop, L, stride, n_mels = 16000, 512, 160, 16000, 160, 40
    p = batch._mel_params(eng.lib, sr, fl, hop, True, "hann", n_mels, 0.0, None, 2.0)
    T = eng.frame_count(L, fl, hop)
    n_units = G31 // (n_mels * T) + 64
    total = (n_units - 1) * stride + L
    need_device_bytes(n_units * n_mels * T * 4 + total * 4 + (2 << 30))
    y = long_input(total, sr, seed=12)
    out = torch.empty((n_units, n_mels, T), dtype=torch.float32, device="cuda")
    try:
        eng.mel_spectrogram_dev(y.data_ptr(), eng.units_clips(n_units, L, total_len=total, stride=stride), p, True, out.data_ptr())
        torch.cuda.synchronize()
        assert eng.lib.dll.syg_debug_last_features_resident() == 0
        one = torch.empty((1, n_mels, T), dtype=torch.float32, device="cuda")

        def single(u):
            eng.mel_spectrogram_dev(y.data_ptr() + 4 * u * stride, eng.units_clips(1, L), p, True, one.data_ptr())
            torch.cuda.synchronize()
            return one[0].cpu().numpy()

        last_units_equal(eng, single, lambda u: out[u].cpu().numpy(), n_units)
        for u in (0, 1):
            assert np.array_equal(single(u), out[u].cpu().numpy()), f"unit {u}"
        u = n_units - 1
        ref = reference(y[u * stride:u * stride + L].cpu().numpy(), sr, fl, hop, n_mels, {}, True)
        assert np.abs(out[u].cpu().numpy() - ref).max() <= DB_TOL
    finally:
        del y, out
        torch.cuda.empty_cache()
