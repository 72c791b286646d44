"""Per-channel forms of the PCM ingest: syg_ingest_pcm_channels (load_audio(mono=False) on the device), and the Welch PSDs and
segment vectors of every (unit, channel) of a host PCM payload in one call (syg_psd_welch_host_pcm_channels,
syg_segment_vectors_host_pcm_channels, batch.channel_psd / channel_vectors).

Every per-channel result must equal, bit for bit, the float32 host form called on that channel's samples alone: the channel forms
only change where the samples come from (one plane per channel, addressed by a per-chunk unit table), never the kernels that run.
"""
import ctypes
import wave

import numpy as np
import pytest

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth

FORMATS = [_ffi.PCM_U8, _ffi.PCM_S16, _ffi.PCM_S24, _ffi.PCM_S32, _ffi.PCM_F32]
SENTINEL = np.float32(-12345.5)


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


def _is_emu(eng):
    return getattr(eng, "test_backend", None) == "emu"


def _dev(eng, *arrays):
    """'Device' copies: CUDA tensors on the B200, the arrays themselves on the emulator (whose device memory is host memory)."""
    if _is_emu(eng):
        hold = [np.ascontiguousarray(a) for a in arrays]
        return hold, [h.ctypes.data for h in hold]
    import torch
    hold = [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]
    return hold, [h.data_ptr() for h in hold]


def _host(h):
    if isinstance(h, np.ndarray):
        return h
    import torch
    torch.cuda.synchronize()
    return h.cpu().numpy()


def _payload(fmt, channels, frames, seed):
    """Random interleaved payload bytes including the extreme codes of the format (negative s24 codes need sign extension)."""
    rng = np.random.default_rng(seed)
    n = frames * channels
    if fmt == _ffi.PCM_U8:
        x = rng.integers(0, 256, n).astype(np.uint8)
        x[:3] = np.array([0, 255, 128], dtype=np.uint8)[: x[:3].size]
        return x
    if fmt == _ffi.PCM_S16:
        x = rng.integers(-32768, 32768, n).astype("<i2")
        x[:4] = np.array([-32768, 32767, 0, -1])[: x[:4].size]
        return x.view(np.uint8)
    if fmt == _ffi.PCM_S24:
        v = rng.integers(-(1 << 23), 1 << 23, n).astype(np.int64)
        v[:4] = np.array([-(1 << 23), (1 << 23) - 1, 0, -1])[: v[:4].size]
        b = np.empty((n, 3), dtype=np.uint8)
        b[:, 0], b[:, 1], b[:, 2] = v & 255, (v >> 8) & 255, (v >> 16) & 255
        return b.reshape(-1)
    if fmt == _ffi.PCM_S32:
        x = rng.integers(-(1 << 31), 1 << 31, n).astype("<i4")
        x[:4] = np.array([-(1 << 31), (1 << 31) - 1, 0, -1])[: x[:4].size]
        return x.view(np.uint8)
    x = (rng.standard_normal(n) * 10.0 ** rng.integers(-4, 1, n)).astype("<f4")
    return x.view(np.uint8)


def _quantise(y, fmt):
    """Float signal [channels, n] in [-1, 1) -> interleaved payload bytes of format fmt."""
    inter = np.ascontiguousarray(y.T)
    if fmt == _ffi.PCM_S16:
        return np.clip(np.round(inter * 32768), -32768, 32767).astype("<i2").reshape(-1).view(np.uint8)
    if fmt == _ffi.PCM_S24:
        v = np.clip(np.round(inter * (1 << 23)), -(1 << 23), (1 << 23) - 1).astype(np.int64).reshape(-1)
        b = np.empty((v.size, 3), dtype=np.uint8)
        b[:, 0], b[:, 1], b[:, 2] = v & 255, (v >> 8) & 255, (v >> 16) & 255
        return b.reshape(-1)
    if fmt == _ffi.PCM_F32:
        return inter.astype("<f4").reshape(-1).view(np.uint8)
    raise ValueError(fmt)


def _recording(fmt, channels, frames, sr, seed):
    """Payload bytes of `channels` different synthetic channels and their float32 planes [channels, frames] as the oracle reads them."""
    y = np.stack([0.7 * synth.mixture(frames, sr, seed=seed + c) for c in range(channels)])
    raw = _quantise(y, fmt)
    return raw, np.ascontiguousarray(orc.load_audio_payload(raw, fmt, channels, mono=False).reshape(channels, frames), dtype=np.float32)


def _units(eng, frames, sr, win_sec, overlap, pad=True):
    seg_len, _, starts, valid = eng.lib.segment_table(frames, sr, win_sec, overlap, pad)
    return eng.units_table(starts.ctypes.data, valid.ctypes.data, len(starts), seg_len, frames), (starts, valid), seg_len


# ---------------------------------------------------------------------------------------------- 1. planar ingest
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("channels", [1, 2, 3, 8, 17, 64])
def test_ingest_channels_bit_exact(eng, fmt, channels):
    """syg_ingest_pcm_channels == soundfile's float32 read per channel, bit for bit; the pad words between the planes (pitch =
    frames rounded up to 4) stay untouched.  Every payload also runs from a device pointer 1-15 bytes past an aligned one."""
    bps = _ffi.PCM_BYTES[fmt]
    for frames in (0, 1, 7, 1000, 4099):
        raw = _payload(fmt, channels, frames, seed=fmt * 100 + channels + frames)
        ref = orc.load_audio_payload(raw, fmt, channels, mono=False).reshape(channels, frames).astype(np.float32)
        pitch = _ffi.plane_pitch(frames)
        assert pitch % 4 == 0 and frames <= pitch < frames + 4
        for off in (0, 1 + (channels * 7 + fmt + frames) % 15):
            buf = np.zeros(raw.size + 32, dtype=np.uint8)
            buf[off:off + raw.size] = raw
            out = np.full(channels * pitch + 8, SENTINEL, dtype=np.float32)
            hold, (praw, pout) = _dev(eng, buf, out)
            eng.ingest_pcm_channels_dev(praw + off, fmt, channels, frames, pout)
            got = _host(hold[1])
            planes = got[:channels * pitch].reshape(channels, pitch)
            assert planes[:, :frames].tobytes() == ref.tobytes(), (fmt, channels, frames, off, bps)
            assert (planes[:, frames:] == SENTINEL).all() and (got[channels * pitch:] == SENTINEL).all(), (fmt, channels, frames, off)


# ---------------------------------------------------------------------------------------------- 2. Welch per channel
WELCH_CASES = [
    # (fmt, channels, sr, window sec, overlap, frames, nperseg, noverlap, nfft, expected kernel)
    (_ffi.PCM_S16, 5, 8000, 0.25, 0.0, 8000 + 777, 1024, 512, 1024, _ffi.WELCH_WARP),       # zero-padded last window
    (_ffi.PCM_S24, 3, 8000, 0.6, 0.5, 8000, 4096, 2048, 4096, _ffi.WELCH_BLOCK),             # 50 % overlapping windows
    (_ffi.PCM_F32, 4, 8000, 0.25, 0.5, 5000, 1000, 500, 1000, _ffi.WELCH_MIXED),
    (_ffi.PCM_S16, 1, 8000, 0.25, 0.0, 6100, 256, 128, 256, _ffi.WELCH_WARP),                # one channel: the mono path
]


def _welch_ref(eng, planes, units, args):
    """syg_psd_welch_host_f32 on each channel's float32 samples alone, with the same units; and the kernel each call reported."""
    psd, st, paths = [], [], set()
    for y in planes:
        p, s = eng.psd_welch_host(y, units, *args, stats=True)
        psd.append(p)
        st.append(s)
        paths.add(eng.lib.dll.syg_debug_last_welch_path())
    return np.stack(psd, axis=1), np.stack(st, axis=1), paths


@pytest.mark.parametrize("case", range(len(WELCH_CASES)))
def test_welch_channels_equal_mono_path(eng, case):
    fmt, ch, sr, win, ov, frames, nperseg, nov, nfft, path = WELCH_CASES[case]
    raw, planes = _recording(fmt, ch, frames, sr, seed=40 + case)
    units, keep, seg_len = _units(eng, frames, sr, win, ov)
    args = (sr, 0, nperseg, nov, nfft, True, 0)
    psd, st = eng.psd_welch_host_pcm_channels(raw.ctypes.data, fmt, ch, units, *args, stats=True)
    got_path = eng.lib.dll.syg_debug_last_welch_path()
    ref_psd, ref_st, ref_paths = _welch_ref(eng, planes, units, args)
    assert got_path == path and ref_paths == {path}
    assert psd.shape == (units.n_units, ch, nfft // 2 + 1) and st.shape == (units.n_units, ch, 3)
    assert psd.tobytes() == ref_psd.tobytes() and st.tobytes() == ref_st.tobytes()
    if ch == 1:                                  # the existing mono path: the PCM payload mixed down (one channel: unchanged)
        mono = eng.psd_welch_host(orc.load_audio_payload(raw, fmt, 1).astype(np.float32), units, *args)
        assert psd[:, 0].tobytes() == mono.tobytes()
    if case in (0, 1):                           # the float64 oracle, at the tolerances of test_parity_cabi.py
        starts, valid = keep
        for u in (0, len(starts) - 1):
            for c in (0, ch - 1):
                seg = np.zeros(seg_len)
                seg[:valid[u]] = planes[c, starts[u]:starts[u] + valid[u]]
                _, ref = orc.compute_psd_welch(seg, fs=sr, nperseg=nperseg, noverlap=nov, nfft=nfft)
                assert (np.abs(psd[u, c] - ref) <= 1e-4 * ref + 2e-6 * ref.max()).all(), (u, c)


# ---------------------------------------------------------------------------------------------- 3. segment vectors per channel
CFG4_FEATURES = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]


FL, HOP, SR_V = 512, 128, 16000


def _ws_per_window(T, n_mels, n_bands, channels):
    """Workspace bytes of one window across its channels, as feat_ws (syg_api.cu) carves a feature unit: unit maxima, mel energies
    [T][n_mels], contrast peaks / valleys [T][2 (n_bands + 1)], each rounded up to 256 bytes, then 256 spare bytes."""
    al = lambda b: (b + 255) // 256 * 256
    return channels * (al(16) + al(T * n_mels * 4) + al(T * 2 * (n_bands + 1) * 4 if n_bands else 0) + 256)


def _chunks(n, ws_window, limit):
    """Windows per chunk of the channel form and the chunk sizes: the workspace limit over the workspace of a window's channels, and
    at most half the windows (two lanes); the sample and output budgets are far from binding here."""
    k = min((n + 1) // 2, max(1, limit // ws_window))
    return k, [min(k, n - w) for w in range(0, n, k)]


def _vectors_case(eng, features, agg, min_groups, fp=None, fmt=_ffi.PCM_S16, ch=3):
    """Both limits, with 21 windows of 0.5 s (50 % overlap): the default limit cuts two chunks of at most 11 windows (the two-lane
    rule), 1 MiB cuts at least three smaller ones (the workspace of a window's channels), so a lane is reused and the cut moves."""
    frames = 5 * SR_V + 3001
    raw, planes = _recording(fmt, ch, frames, SR_V, seed=7)
    units, _, seg_len = _units(eng, frames, SR_V, 0.5, 0.5)
    n = int(units.n_units)
    p = _ffi.make_params(eng.lib, SR_V, features, FL, HOP, feature_params=fp)
    T = eng.frame_count(seg_len, FL, HOP)
    n_mels = (fp or {}).get("mfcc", {}).get("n_mels", 128) if "mfcc" in features else 0
    ws_window = _ws_per_window(T, n_mels, 6 if "spectral_contrast" in features else 0, ch)
    ids = [_ffi.AGG_IDS[agg]] * eng.rows(p) if isinstance(agg, str) else [agg[i % len(agg)] for i in range(eng.rows(p))]
    gpu = not _is_emu(eng)
    eng.lib.dll.syg_debug_set_resident_min_groups(min_groups)
    eng.profile_enable(True)
    try:
        results, cuts = [], []
        for limit in (1 << 30, 1 << 20):
            k, sizes = _chunks(n, ws_window, limit)
            cuts.append(k)
            eng.set_workspace_limit(limit)
            eng.profile_read(reset=True)
            got = eng.segment_vectors_host_pcm_channels(raw.ctypes.data, fmt, ch, units, p, ids)
            frame_launches = eng.profile_read(reset=True)["frame"][1]
            kinds = (eng.lib.dll.syg_debug_last_features_resident(), eng.lib.dll.syg_debug_last_feature_kernel())
            fin = eng.lib.last_finalize()
            if gpu:                                   # one frame-kernel launch per chunk (the emulator's events count nothing)
                assert frame_launches == len(sizes), (limit, frame_launches, sizes)
            if kinds[0] == 0:                         # the last chunk's finalize: its (window, channel) units' frames in 32-frame tiles
                assert fin[0] == 32 and fin[2] == (sizes[-1] * ch * T + 31) // 32, (limit, fin, sizes)
            ref = np.stack([eng.segment_vectors_host(planes[c].ctypes.data, units, p, ids) for c in range(ch)], axis=1)
            ref_kinds = (eng.lib.dll.syg_debug_last_features_resident(), eng.lib.dll.syg_debug_last_feature_kernel())
            assert got.shape == (n, ch, eng.rows(p))
            assert kinds == ref_kinds, (limit, kinds, ref_kinds)
            assert got.tobytes() == ref.tobytes(), limit
            results.append((got, kinds))
        assert n >= 20 and cuts[1] < cuts[0] == (n + 1) // 2 and len(_chunks(n, ws_window, 1 << 20)[1]) >= 3, (n, cuts)
        return results
    finally:
        eng.profile_enable(False)
        eng.profile_read(reset=True)
        eng.set_workspace_limit(1 << 30)
        eng.lib.dll.syg_debug_set_resident_min_groups(-1)


@pytest.mark.parametrize("agg", ["mean", "std", "median", "min", "max"])
def test_vectors_channels_equal_mono_path_cfg4(eng, agg):
    """cfg4's feature request (two-kernel path with finalize) per channel equals syg_segment_vectors_host_f32 on each channel, at
    both limits, whatever the cut."""
    (a, ka), (b, kb) = _vectors_case(eng, CFG4_FEATURES, agg, min_groups=1 << 30)
    assert ka[0] == 0 and a.tobytes() == b.tobytes()


def test_vectors_channels_resident_epilogue(eng):
    """An MFCC-only request with the resident minimum lowered: both calls keep their units on chip (resident epilogue)."""
    (a, ka), (b, kb) = _vectors_case(eng, ["mfcc"], [0, 1, 3, 4], min_groups=1, fp={"mfcc": {"n_mels": 128}}, fmt=_ffi.PCM_S24, ch=4)
    assert ka == (1, _ffi.FK_RESIDENT) and a.tobytes() == b.tobytes()


# ---------------------------------------------------------------------------------------------- 4. errors
def test_channel_forms_errors(eng):
    """Each bad argument returns its code and leaves a sentinel-filled output untouched."""
    sr, frames, ch = 8000, 4000, 2
    raw, _ = _recording(_ffi.PCM_S16, ch, frames, sr, seed=3)
    units, keep, _ = _units(eng, frames, sr, 0.25, 0.0)
    n = int(units.n_units)
    psd = np.full((n, ch, 129), SENTINEL, np.float32)
    st = np.full((n, ch, 3), SENTINEL, np.float32)
    p = _ffi.make_params(eng.lib, sr, ["rms_energy"], 256, 64)
    agg = (ctypes.c_int32 * 1)(0)
    vec = np.full((n, ch, 1), SENTINEL, np.float64)
    d = eng.lib.dll

    def welch(ptr=raw.ctypes.data, fmt=_ffi.PCM_S16, c=ch, u=units, nfft=256, out=psd.ctypes.data):
        return d.syg_psd_welch_host_pcm_channels(eng._h, ptr, fmt, c, ctypes.byref(u), float(sr), 0, 256, 128, nfft, 1, 0, out,
                                                 st.ctypes.data)

    def vectors(ptr=raw.ctypes.data, fmt=_ffi.PCM_S16, c=ch, u=units, a=agg):
        return d.syg_segment_vectors_host_pcm_channels(eng._h, ptr, fmt, c, ctypes.byref(u), ctypes.byref(p),
                                                       ctypes.addressof(a) if a is not None else None, vec.ctypes.data)

    starts, valid = keep
    bad_starts = starts.copy()
    bad_starts[-1] = frames - int(valid[-1]) + 1                      # the last unit's samples run one frame past the payload
    outside = eng.units_table(bad_starts.ctypes.data, valid.ctypes.data, n, units.unit_len, frames)
    for c in (0, 65, -1):
        assert welch(c=c) == _ffi.SYG_E_BADARG and vectors(c=c) == _ffi.SYG_E_BADARG
    for fmt in (-1, 5):
        assert welch(fmt=fmt) == _ffi.SYG_E_BADARG and vectors(fmt=fmt) == _ffi.SYG_E_BADARG
    assert welch(ptr=None) == _ffi.SYG_E_BADARG and vectors(ptr=None) == _ffi.SYG_E_BADARG
    assert welch(out=None) == _ffi.SYG_E_BADARG and vectors(a=None) == _ffi.SYG_E_BADARG
    assert welch(u=outside) == _ffi.SYG_E_BADARG and vectors(u=outside) == _ffi.SYG_E_BADARG
    assert welch(nfft=1006) == _ffi.SYG_E_UNSUPPORTED                # 2 * 503: the plan error of the float32 form
    assert (psd == SENTINEL).all() and (st == SENTINEL).all() and (vec == SENTINEL).all()
    assert welch(u=eng.units_clips(0, 4000)) == _ffi.SYG_OK and vectors(u=eng.units_clips(0, 4000)) == _ffi.SYG_OK
    assert (psd == SENTINEL).all() and (vec == SENTINEL).all()
    out = np.full(64, SENTINEL, np.float32)
    hold, (praw, pout) = _dev(eng, raw, out)
    for fmt, c in ((_ffi.PCM_S16, 0), (_ffi.PCM_S16, 65), (7, 2)):
        assert d.syg_ingest_pcm_channels(eng._h, praw, fmt, c, 8, pout, None) == _ffi.SYG_E_BADARG
    assert d.syg_ingest_pcm_channels(eng._h, None, _ffi.PCM_S16, 2, 8, pout, None) == _ffi.SYG_E_BADARG
    assert (_host(hold[1]) == SENTINEL).all()
    # preallocated results the library would write past or scatter into are refused before the call
    wel = (float(sr), 0, 256, 128, 256)
    for bad in (np.empty((n, ch, 128), np.float32), np.empty((n, ch, 129), np.float64), np.empty((n, 129, ch), np.float32).transpose(0, 2, 1)):
        with pytest.raises(ValueError):
            eng.psd_welch_host_pcm_channels(raw.ctypes.data, _ffi.PCM_S16, ch, units, *wel, out=(bad, None))
    with pytest.raises(ValueError):
        eng.psd_welch_host_pcm_channels(raw.ctypes.data, _ffi.PCM_S16, ch, units, *wel, stats=True, out=(psd, st[:, :1]))
    with pytest.raises(ValueError):
        eng.segment_vectors_host_pcm_channels(raw.ctypes.data, _ffi.PCM_S16, ch, units, p, [0], out=vec[:-1])
    assert (psd == SENTINEL).all() and (st == SENTINEL).all() and (vec == SENTINEL).all()


# ---------------------------------------------------------------------------------------------- 5. GPU: one launch per chunk
@pytest.mark.gpu
def test_one_launch_per_chunk_gpu():
    """64 channels x 50 one-second windows at 25.6 kHz: 328 MB of float32 samples.  A chunk takes 128 MiB of samples, 20 windows of
    64 channels (less than the two-lane cap of 25 windows), so the call cuts chunks of 20, 20 and 10 windows (1280, 1280 and 640
    (window, channel) units), reuses a lane for the third, and issues one ingest and one Welch launch per chunk."""
    eng = get_engine("gpu")
    sr, ch, sec = 25600, 64, 50
    y = synth.long_signal(ch * sec * sr, sr, seed=5).reshape(ch, sec * sr) * 0.5
    raw = _quantise(y, _ffi.PCM_S16)
    planes = orc.load_audio_payload(raw, _ffi.PCM_S16, ch, mono=False).astype(np.float32)
    units = eng.units_clips(sec, sr)
    args = (sr, 0, 1024, 512, 1024, True, 0)
    eng.profile_enable(True)
    try:
        eng.profile_read(reset=True)
        psd, st = eng.psd_welch_host_pcm_channels(raw.ctypes.data, _ffi.PCM_S16, ch, units, *args, stats=True)
        prof = eng.profile_read(reset=True)
    finally:
        eng.profile_enable(False)
        eng.profile_read(reset=True)
    assert ((128 << 20) // (sr * 4 * ch), (sec + 1) // 2) == (20, 25)
    assert prof["other"][1] == 3 and prof["welch"][1] == 3, prof
    ref_psd, ref_st, _ = _welch_ref(eng, planes, units, args)
    assert psd.tobytes() == ref_psd.tobytes() and st.tobytes() == ref_st.tobytes()


# ---------------------------------------------------------------------------------------------- 6. GPU: Python on a WAV file
def _write_wav_s24(path, raw, sr, channels):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(channels)
        w.setsampwidth(3)
        w.setframerate(sr)
        w.writeframes(bytes(raw))


@pytest.mark.gpu
def test_channel_psd_wav_gpu(tmp_path):
    from sygnals_b200 import batch
    from sygnals_b200.core.audio import io as sio
    eng = get_engine("gpu")
    sr, ch, frames = 25600, 6, int(3.4 * 25600)
    raw, planes = _recording(_ffi.PCM_S24, ch, frames, sr, seed=21)
    path = tmp_path / "six.wav"
    _write_wav_s24(path, raw, sr, ch)
    r = batch.channel_psd(path)
    units, (starts, valid), _ = _units(eng, frames, sr, 1.0, 0.0)
    ref_psd, ref_st, _ = _welch_ref(eng, planes, units, (sr, 0, 1024, 512, 1024, True, 0))
    assert r["psd"].shape == (4, ch, 513) and r["sample_rate"] == sr
    assert np.array_equal(r["starts"], starts) and np.array_equal(r["valid"], valid)
    assert np.allclose(r["freqs"], np.arange(513) * sr / 1024)
    assert r["psd"].tobytes() == ref_psd.tobytes() and r["stats"].tobytes() == ref_st.tobytes()
    r2 = batch.channel_psd(batch.Payload(raw, _ffi.PCM_S24, ch, sr), stats=False)
    assert r2["stats"] is None and r2["psd"].tobytes() == ref_psd.tobytes()
    names, vec = batch.channel_vectors(path, 1.0, ["mfcc", "rms_energy"], aggregation="max")
    p = _ffi.make_params(eng.lib, sr, ["mfcc", "rms_energy"])
    ids = [_ffi.AGG_IDS["max"]] * eng.rows(p)
    ref = np.stack([eng.segment_vectors_host(planes[c].ctypes.data, units, p, ids) for c in range(ch)], axis=1)
    assert names[0] == "mfcc_0" and vec.shape == (4, ch, 14) and vec.tobytes() == ref.tobytes()
    eng.profile_enable(True)
    try:
        eng.profile_read(reset=True)
        y, got_sr = sio.load_audio(path, mono=False)
        prof = eng.profile_read(reset=True)
    finally:
        eng.profile_enable(False)
        eng.profile_read(reset=True)
    assert got_sr == sr and y.dtype == np.float64 and y.shape == (ch, frames)
    assert np.array_equal(y, orc.load_audio_payload(raw, _ffi.PCM_S24, ch, mono=False))
    assert prof["other"][1] == 1, prof
