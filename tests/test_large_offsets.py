"""Sample buffers, unit offsets and outputs past 2^31 and 2^32 elements.

One long recording is one sample buffer and units are framed by index (DESIGN.md section 3): 13.5 h at 44.1 kHz is 2^31
samples, 27 h is 2^32, and outputs (a 10 h STFT, a batch of a million overlapping units) cross 2^31 elements sooner.  Every
entry point is run here on units that sit across, just below, just above and well past element 2^31 and 2^32, with frames and
zero tails that cross the boundaries, and each result is checked twice:

* twin bit-equality: the same samples at a small offset with the same alignment modulo 16 bytes make the launcher pick the
  same kernel (the debug getters must agree), so the result must be identical bit for bit; an index that wraps reads other
  samples and breaks it;
* parity with the float64 oracle at the tolerances of test_parity_cabi.py.

The host buffers are np.zeros arrays of up to 2^32 + 2^18 samples whose pages are mapped only where a window is written, so the
emulator leg (whose device memory is host memory) and the host forms cost a few MB.  On the GPU the device forms copy the windows
into torch.zeros buffers of up to 17 GB; a test skips, saying so, when the device has less free memory than it needs plus 4 GB.
The outputs past 2^31 elements are written in full, so those cases run on the GPU only."""
import contextlib

import numpy as np
import pytest

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi, batch
from sygnals_b200.utils import synth
from test_parity_cabi import _dev_buffers, _host, check_rows, oracle_rows, power_close

G31, G32 = 1 << 31, 1 << 32
N_BIG = G32 + (1 << 18)            # samples of the lazily zeroed recording
REGION = 1 << 16                   # written samples on each side of 0, 2^31 and 2^32
MARGIN = 4 << 30                   # free device memory left to the other users of a shared GPU
AGG = ["mean", "std", "median", "min", "max"]
CFG4 = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]

# name -> (sr, frame_length, hop, features, feature_params): one request per feature-kernel family
FEATURES = {
    "resident512": (16000, 512, 160, ["mfcc", "rms_energy", "spectral_centroid"], {"mfcc": {"n_mels": 40}}),
    "warp1024": (22050, 1024, 256, CFG4, {"mfcc": {"n_mels": 40}}),
    "spec44kl": (44100, 2048, 512, CFG4, None),                  # the cfg4 request: Spec44kL specialisation
    "block4096": (48000, 4096, 1024, ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy"], None),
    "mixed1000": (16000, 1000, 250, ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy"], {"mfcc": {"n_mels": 40}}),
    "time_extra": (22050, 1024, 256, ["zero_crossing_rate", "skewness", "kurtosis", "signal_entropy", "rms_energy",
                                      "spectral_centroid"], None),
}


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


def on_gpu(eng):
    return eng.test_backend == "gpu"


def need_device_bytes(nbytes):
    import torch
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + MARGIN:
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory plus a 4 GiB margin; the shared GPU has "
                    f"{free / 2**30:.1f} GiB free")


class Lazy:
    """float32 (or any dtype) buffer that is zero except for the windows written into it: numpy maps the pages of np.zeros only
    where they are written, so a buffer of 2^32 samples costs the size of its windows."""

    def __init__(self, n, dtype=np.float32):
        self.y = np.zeros(n, dtype)
        self.windows = []

    def put(self, at, x):
        self.y[at:at + len(x)] = x
        self.windows.append((at, at + len(x)))


def recording(sr, seed=1):
    """N_BIG samples: a signal in [0, REGION), around 2^31 and from 2^32 - REGION to the end, zeros elsewhere."""
    b = Lazy(N_BIG)
    for i, (lo, hi) in enumerate([(0, REGION), (G31 - REGION, G31 + REGION), (G32 - REGION, N_BIG)]):
        b.put(lo, synth.mixture(hi - lo, sr, seed=seed + i))
    return b


@contextlib.contextmanager
def device(eng, *bufs):
    """Device pointers to copies of Lazy buffers: the buffers themselves on the emulator; on the GPU torch.zeros buffers with the
    windows copied in, freed on exit."""
    if not on_gpu(eng):
        yield [b.y.ctypes.data for b in bufs]
        return
    import torch
    need_device_bytes(sum(b.y.nbytes for b in bufs))
    held = []
    try:
        for b in bufs:
            t = torch.zeros(b.y.nbytes, dtype=torch.uint8, device="cuda")
            raw = b.y.view(np.uint8)
            for lo, hi in b.windows:
                k = b.y.itemsize
                t[lo * k:hi * k].copy_(torch.from_numpy(raw[lo * k:hi * k]))
            held.append(t)
        t = None
        yield [h.data_ptr() for h in held]
        torch.cuda.synchronize()
    finally:
        held.clear()
        t = None
        torch.cuda.empty_cache()


def sync(eng):
    if on_gpu(eng):
        import torch
        torch.cuda.synchronize()


def getters(eng):
    d = eng.lib.dll
    return (d.syg_debug_last_stft_path(), d.syg_debug_last_features_resident(), d.syg_debug_last_mel_form(),
            d.syg_debug_last_feature_frames())


# ------------------------------------------------------------------------------------------------ unit geometry
def geometry(kind, L):
    """(starts, valid, total_len, stride) of the units of one call.

    table / table_total: eight units in buffer order (the host forms' two chunks stay near 2^31 and near 2^32): ending at 2^31,
    frames across 2^31, a valid part below 2^31 with its zero tail across it, starting at 2^31; frames across 2^32, a zero tail
    across 2^32, an odd offset past 2^32, and a last unit whose valid part ends at total_len.  ``table`` passes the valid lengths,
    ``table_total`` derives them from total_len.
    stride_cross / stride_tail: analytic geometry, unit 1 across 2^31 / past 2^32 with its valid part ending at total_len."""
    if kind in ("table", "table_total"):
        units = [(G31 - L, L), (G31 - L // 2 - 1, L), (G31 - L // 2 + 3, L // 3), (G31, L),
                 (G32 - L // 2 + 1, L), (G32 - 2 * (L // 3) + 1, L // 3), (G32 + 12345, L), (G32 + 40001, L // 2 + 3)]
        starts = [s for s, _ in units]
        if kind == "table":
            return starts, [v for _, v in units], N_BIG, None
        return starts, None, starts[-1] + units[-1][1], None
    h = 4 * (L // 8)                    # multiples of 4 keep the STFT ring kernel's layout conditions
    if kind == "stride_cross":
        s = G31 - h - 4
        return [0, s], None, N_BIG, s
    s = G32 + 12
    return [0, s], None, s + h + 4, s


def valid_of(starts, valid, total, L):
    return [min(max(total - s, 0), L) if valid is None else v for s, v in zip(starts, valid or starts)]


def twin(y, starts, valid, total, stride, L):
    """The same units rebased near 0, each start congruent to its original modulo 4 samples (16 bytes): (y2, starts2, total2,
    stride2).  Analytic units stay analytic (stride2 congruent to stride), and the last unit keeps its distance to total_len."""
    n = len(starts)
    if stride is not None:
        stride2 = L + 64 + (stride - L - 64) % 4
        s2 = [u * stride2 for u in range(n)]
    else:
        stride2 = None
        s2 = [4096 + u * (L + 68) + (s - 4096 - u * (L + 68)) % 4 for u, s in enumerate(starts)]
    tail = total - starts[-1]
    if tail > L:
        tail = L + 64 + (tail - L - 64) % 4
    y2 = np.zeros(s2[-1] + max(tail, L) + 64, y.dtype)
    for a, b in zip(starts, s2):
        w = y[a:a + L]
        y2[b:b + len(w)] = w
    return y2, s2, s2[-1] + tail, stride2


class Units:
    """syg_units of one geometry; ``dev`` puts the start / valid tables in device memory."""

    def __init__(self, eng, starts, valid, total, stride, L, dev=False):
        if stride is not None:
            self.u = eng.units_clips(len(starts), L, total_len=total, stride=stride)
            return
        st = np.asarray(starts, np.int64)
        va = np.asarray(valid, np.int32) if valid is not None else None
        if dev:
            self.hold, ptrs = _dev_buffers(eng, *([st] if va is None else [st, va]))
        else:
            self.hold = [st, va]
            ptrs = [st.ctypes.data] + ([va.ctypes.data] if va is not None else [])
        self.u = eng.units_table(ptrs[0], ptrs[1] if va is not None else 0, len(st), L, total)


def unit_window(y, s, v, L):
    seg = np.zeros(L, np.float32)
    seg[:v] = y[s:s + v]
    return seg


GEOMS = ["table", "table_total", "stride_cross", "stride_tail"]


# ------------------------------------------------------------------------------------------------ features / segment vectors
def run_features(eng, p, L, big_ptr, big_y, kind, agg_ids=None):
    """host and device forms on the recording and on its twin: {form: (big result, twin result, getters big, getters twin)}"""
    starts, valid, total, stride = geometry(kind, L)
    y2, s2, total2, stride2 = twin(big_y, starts, valid, total, stride, L)
    rows, T = eng.rows(p), eng.frame_count(L, p.frame_length, p.hop_length, p.center)
    res = {}
    for form in ("host", "dev"):
        pair, gets = [], []
        for y, ptr, st, tl, sd in ((big_y, big_ptr, starts, total, stride), (y2, None, s2, total2, stride2)):
            u = Units(eng, st, valid, tl, sd, L, dev=form == "dev")
            if form == "host":
                out = (eng.features_host(y, u.u, p) if agg_ids is None else
                       eng.segment_vectors_host(y.ctypes.data, u.u, p, agg_ids))
                gets.append(getters(eng))
            else:
                shape, dt = ((len(st), rows, T), np.float32) if agg_ids is None else ((len(st), rows), np.float64)
                hold, (po,) = _dev_buffers(eng, np.zeros(shape, dt))
                if ptr is None:
                    hy, (ptr,) = _dev_buffers(eng, y)
                if agg_ids is None:
                    eng.features_dev(ptr, u.u, p, po)
                else:
                    eng.segment_vectors_dev(ptr, u.u, p, agg_ids, po)
                gets.append(getters(eng))
                sync(eng)
                out = _host(eng, hold[0])
            pair.append(out)
        res[form] = (pair[0], pair[1], gets[0], gets[1])
    return res, starts, valid_of(starts, valid, total, L)


@contextlib.contextmanager
def resident(eng, on):
    eng.lib.dll.syg_debug_set_resident_min_groups(1 if on else 1 << 30)
    try:
        yield
    finally:
        eng.lib.dll.syg_debug_set_resident_min_groups(-1)


@pytest.mark.parametrize("case,center", [(c, True) for c in FEATURES] + [("time_extra", False), ("warp1024", False)])
def test_features_past_2g(eng, case, center):
    sr, fl, hop, feats, fp = FEATURES[case]
    L = fl + 3 * hop + 5
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, center=center, feature_params=fp)
    big = recording(sr, seed=fl + hop)
    names = batch.feature_row_names(feats, fp)
    with device(eng, big) as (py,), resident(eng, case == "resident512"):
        for kind in GEOMS:
            res, starts, valid = run_features(eng, p, L, py, big.y, kind)
            refs = [oracle_rows(unit_window(big.y, s, v, L), sr, feats, fl, hop, fp, center=center) for s, v in zip(starts, valid)]
            for form, (got, got2, g, g2) in res.items():
                assert g == g2, f"{kind} {form}: the twin took another kernel path {g} != {g2}"
                assert g[1] == (case == "resident512"), f"{kind} {form}: resident epilogue {g[1]}"
                assert g[3] == len(starts) * got.shape[2]
                assert np.array_equal(got, got2, equal_nan=True), f"{kind} {form}: differs from the same units near 0"
                for u, (rn, ref) in enumerate(refs):
                    assert rn == names
                    check_rows(names, got[u], ref, bin_hz=sr / fl, nyq=sr / 2)


@pytest.mark.parametrize("case", ["warp1024", "block4096"])
def test_segment_vectors_past_2g(eng, case):
    """Every aggregation (rows cycle through mean / std / median / min / max) == the oracle's formatter on the frame features."""
    sr, fl, hop, feats, fp = FEATURES[case]
    L = fl + 3 * hop + 5
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    names = batch.feature_row_names(feats, fp)
    ids = [r % len(AGG) for r in range(len(names))]
    how = {n: AGG[i] for n, i in zip(names, ids)}
    big = recording(sr, seed=7)
    with device(eng, big) as (py,):
        for kind in GEOMS:
            vec, _, _ = run_features(eng, p, L, py, big.y, kind, agg_ids=ids)
            frames, _, _ = run_features(eng, p, L, py, big.y, kind)
            for form in ("host", "dev"):
                v, v2, g, g2 = vec[form]
                assert g == g2 and np.array_equal(v, v2, equal_nan=True), f"{kind} {form}"
                F = frames[form][0]
                for u in range(F.shape[0]):
                    ref = orc.format_feature_vectors_per_segment({n: F[u, r].astype(np.float64) for r, n in enumerate(names)},
                                                                 [(0, F.shape[2])], how)[0]
                    for r, n in enumerate(names):
                        if how[n] in ("median", "min", "max"):
                            assert v[u, r] == ref[r], f"{kind} {form} unit {u} {n}"
                        else:
                            np.testing.assert_allclose(v[u, r], ref[r], rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------------------------------------ STFT
# family -> (n_fft, hop, win_length, pad_mode, out_kind, geometry kinds, expected syg_debug_last_stft_path)
STFT = {
    "ring1024": (1024, 256, 1024, 0, _ffi.OUT_POWER, ["stride_cross", "stride_tail"], 1),
    "ring256": (256, 64, 256, 0, _ffi.OUT_POWER, ["stride_cross", "stride_tail"], 1),
    "warp512": (512, 128, 400, 0, _ffi.OUT_COMPLEX, GEOMS, 2),
    "sub4096": (4096, 1024, 4096, 0, _ffi.OUT_POWER, GEOMS, 4),
    "sub8192": (8192, 2048, 8192, 0, _ffi.OUT_MAGNITUDE, ["table", "stride_tail"], 4),
    "cta4096": (4096, 1024, 3000, 1, _ffi.OUT_COMPLEX, ["table", "stride_tail"], 3),
    "mixed400": (400, 160, 400, 0, _ffi.OUT_POWER, GEOMS, 5),
}


@pytest.mark.parametrize("family", list(STFT))
def test_stft_past_2g(eng, family):
    n_fft, hop, wl, pad, kind_out, kinds, path = STFT[family]
    L = 2 * n_fft + 3 * hop + 4                    # a multiple of 4: the ring kernel's bulk copies need it
    big = recording(22050, seed=n_fft)
    B = 1 + n_fft // 2
    T = eng.frame_count(L, n_fft, hop, True)
    dt = np.complex64 if kind_out == _ffi.OUT_COMPLEX else np.float32
    with device(eng, big) as (py,):
        for kind in kinds:
            starts, valid, total, stride = geometry(kind, L)
            if pad == 1 and valid is not None:
                valid = [max(v, n_fft // 2 + 1) for v in valid]        # reflect padding needs more than n_fft / 2 valid samples
            y2, s2, total2, stride2 = twin(big.y, starts, valid, total, stride, L)
            outs = {}
            for form in ("host", "dev"):
                for tag, y, ptr, st, tl, sd in (("big", big.y, py, starts, total, stride), ("twin", y2, None, s2, total2, stride2)):
                    u = Units(eng, st, valid, tl, sd, L, dev=form == "dev")
                    if form == "host":
                        out = eng.stft_host(y, u.u, n_fft, hop, wl, center=True, pad_mode=pad, out_kind=kind_out)
                    else:
                        hold, (po,) = _dev_buffers(eng, np.zeros((len(st), B, T), dt))
                        if ptr is None:
                            hy, (ptr,) = _dev_buffers(eng, y)
                        eng.stft_dev(ptr, u.u, n_fft, hop, wl, 0, True, pad, kind_out, po)
                        sync(eng)
                        out = _host(eng, hold[0])
                    outs[form, tag] = (out, eng.lib.dll.syg_debug_last_stft_path())
            for form in ("host", "dev"):
                (a, pa), (b, pb) = outs[form, "big"], outs[form, "twin"]
                assert pa == pb == path, f"{kind} {form}: paths {pa} / {pb}, expected {path}"
                assert np.array_equal(a, b), f"{kind} {form}: differs from the same units near 0"
                for u, (s, v) in enumerate(zip(starts, valid_of(starts, valid, total, L))):
                    seg = unit_window(big.y, s, v, L)[:v if pad == 1 else L].astype(np.float64)
                    D = orc.compute_stft(seg, n_fft=n_fft, hop_length=hop, win_length=wl, center=True,
                                         pad_mode="reflect" if pad == 1 else "constant")
                    if pad == 1:                       # reflect padding mirrors inside the valid part: compare its frames
                        D = D[:, :a.shape[2]] if D.shape[1] >= a.shape[2] else D
                        got = a[u][:, :D.shape[1]]
                    else:
                        got = a[u]
                    ref = np.abs(D) ** 2
                    P = np.abs(got.astype(np.complex128)) ** 2 if kind_out != _ffi.OUT_POWER else got.astype(np.float64)
                    if kind_out == _ffi.OUT_MAGNITUDE:
                        P = got.astype(np.float64) ** 2
                    power_close(P, ref)


# ------------------------------------------------------------------------------------------------ Welch
@pytest.mark.parametrize("nperseg,noverlap,nfft", [(1024, 512, 1024), (500, 250, 1000)])
def test_welch_past_2g(eng, nperseg, noverlap, nfft):
    """psd_welch with stats on the warp kernel (1024) and the mixed-radix kernel (nfft 1000)."""
    sr = 25600
    L = 4 * nperseg + 4
    big = recording(sr, seed=nfft)
    with device(eng, big) as (py,):
        for kind in GEOMS:
            starts, valid, total, stride = geometry(kind, L)
            valid = None if valid is None else [max(v, nperseg) for v in valid]       # a unit holds whole Welch segments
            y2, s2, total2, stride2 = twin(big.y, starts, valid, total, stride, L)
            res = {}
            for form in ("host", "dev"):
                for tag, y, ptr, st, tl, sd in (("big", big.y, py, starts, total, stride), ("twin", y2, None, s2, total2, stride2)):
                    u = Units(eng, st, valid, tl, sd, L, dev=form == "dev")
                    if form == "host":
                        res[form, tag] = eng.psd_welch_host(y, u.u, sr, 0, nperseg, noverlap, nfft, True, 0, stats=True)
                        continue
                    hold, (pp, ps) = _dev_buffers(eng, np.zeros((len(st), nfft // 2 + 1), np.float32), np.zeros((len(st), 3), np.float32))
                    if ptr is None:
                        hy, (ptr,) = _dev_buffers(eng, y)
                    eng.psd_welch_dev(ptr, u.u, sr, 0, nperseg, noverlap, nfft, True, 0, pp, ps)
                    sync(eng)
                    res[form, tag] = (_host(eng, hold[0]), _host(eng, hold[1]))
            for form in ("host", "dev"):
                (psd, st_), (psd2, st2) = res[form, "big"], res[form, "twin"]
                assert np.array_equal(psd, psd2) and np.array_equal(st_, st2), f"{kind} {form}"
                for u, (s, v) in enumerate(zip(starts, valid_of(starts, valid, total, L))):
                    seg = unit_window(big.y, s, v, L).astype(np.float64)
                    _, ref = orc.compute_psd_welch(seg, fs=sr, nperseg=nperseg, noverlap=noverlap, nfft=nfft)
                    assert (np.abs(psd[u] - ref) <= 1e-4 * ref + 2e-6 * ref.max()).all(), f"{kind} {form} unit {u}"
                    rms = np.sqrt(np.mean(seg ** 2))
                    np.testing.assert_allclose(st_[u], [rms, np.abs(seg).max() / rms, np.abs(seg).max()], rtol=1e-5)


# ------------------------------------------------------------------------------------------------ ragged batches
RAGGED = (16000, 512, 160, ["mfcc", "spectral_contrast", "rms_energy", "spectral_centroid"], {"mfcc": {"n_mels": 40}})


def ragged_call(eng, y_host, y_dev, starts, lengths, total, p, agg_ids=None):
    """features (or segment vectors) of one ragged batch, host and device form"""
    units = eng.ragged_units(starts, lengths, total)
    foff = eng.lib.ragged_frame_offsets(units, p.frame_length, p.hop_length, p.center)
    if agg_ids is None:
        h = eng.features_ragged_host(y_host, units, p)
        hold, (po,) = _dev_buffers(eng, np.zeros((eng.rows(p), foff[-1]), np.float32))
        eng.features_ragged_dev(y_dev, units, p, po)
    else:
        h = eng.segment_vectors_ragged_host(y_host, units, p, agg_ids)
        hold, (po,) = _dev_buffers(eng, np.zeros((len(starts), eng.rows(p)), np.float64))
        eng.segment_vectors_ragged_dev(y_dev, units, p, agg_ids, po)
    sync(eng)
    return foff, h, _host(eng, hold[0])


def test_ragged_past_2g(eng):
    """Units at 0, across 2^31 and past 2^32 in one call: each unit's columns equal its single-unit call, the same units rebased
    near 0, and the oracle; the segment vectors equal the twin's."""
    sr, fl, hop, feats, fp = RAGGED
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    names = batch.feature_row_names(feats, fp)
    big = recording(sr, seed=5)
    starts = np.array([0, G31 - 1001, G31 - 3, G31 + 6, G32 - 700, G32 + 12345, N_BIG - 2001], np.int64)
    lengths = np.array([3000, 2500, 700, 1, 1500, 2222, 2001], np.int64)
    s2 = np.array([64 + 4096 * i + int(s) % 4 for i, s in enumerate(starts)], np.int64)
    y2 = np.zeros(int(s2[-1] + 4096), np.float32)
    for a, b, n in zip(starts, s2, lengths):
        y2[b:b + n] = big.y[a:a + n]
    ids = [r % len(AGG) for r in range(len(names))]
    with device(eng, big) as (py,):
        foff, h, d = ragged_call(eng, big.y, py, starts, lengths, N_BIG, p)
        hy, (py2,) = _dev_buffers(eng, y2)
        foff2, h2, d2 = ragged_call(eng, y2, py2, s2, lengths, len(y2), p)
        assert np.array_equal(foff, foff2)
        for got in (h, d, h2, d2):
            assert np.array_equal(got, h, equal_nan=True)
        refs, cols = [], []
        for u, (s, n) in enumerate(zip(starts, lengths)):
            seg = big.y[s:s + n]
            one = eng.features_host(seg, eng.units_clips(1, int(n)), p)[0]
            assert np.array_equal(one, h[:, foff[u]:foff[u + 1]], equal_nan=True), f"unit {u} at {s}"
            if n >= fl:
                refs.append(oracle_rows(seg, sr, feats, fl, hop, fp)[1])
                cols.append(h[:, foff[u]:foff[u + 1]])
        # one check over all units: the contrast bar counts entries, and a short unit has few
        check_rows(names, np.concatenate(cols, axis=1), np.concatenate(refs, axis=1), bin_hz=sr / fl, nyq=sr / 2)
        _, v, vd = ragged_call(eng, big.y, py, starts, lengths, N_BIG, p, ids)
        _, v2, vd2 = ragged_call(eng, y2, py2, s2, lengths, len(y2), p, ids)
        for got in (vd, v2, vd2):
            assert np.array_equal(got, v, equal_nan=True)


@pytest.mark.parametrize("span", [G31 - 1, G31, G32 + 5])
def test_ragged_device_chunk_span(eng, span):
    """Two units whose samples span exactly 2^31 - 1 (one chunk of the device form), 2^31 (two chunks: the frame table's starts
    are chunk-relative int32) and more than 2^32: the same columns as each unit alone."""
    sr, fl, hop, feats, fp = RAGGED
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    big = recording(sr, seed=11)
    lengths = np.array([1500, 1300], np.int64)
    a = G31 - 2 * REGION // 3 if span < G32 else 100
    starts = np.array([a, a + span - lengths[1]], np.int64)
    assert starts[1] + lengths[1] - starts[0] == span and starts[1] + lengths[1] <= N_BIG
    with device(eng, big) as (py,):
        foff, h, d = ragged_call(eng, big.y, py, starts, lengths, N_BIG, p)
    assert np.array_equal(h, d, equal_nan=True)
    for u, (s, n) in enumerate(zip(starts, lengths)):
        one = eng.features_host(big.y[s:s + n], eng.units_clips(1, int(n)), p)[0]
        assert np.array_equal(one, d[:, foff[u]:foff[u + 1]], equal_nan=True), f"unit {u}"


def test_ragged_unit_of_2g_samples_is_unsupported(eng):
    """A unit of 2^31 samples: SYG_E_UNSUPPORTED before anything runs (the output stays untouched)."""
    import ctypes as C
    p = _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160)
    y = np.zeros(G31 + 8, np.float32)
    units = eng.ragged_units([4], [G31], len(y))
    out = np.full((13, 8), 7.0, np.float32)
    d, args = eng.lib.dll, (eng._h, y.ctypes.data, C.byref(units), C.byref(p))
    ids = (C.c_int32 * 13)(*([0] * 13))
    for rc in (d.syg_features_ragged_host_f32(*args, out.ctypes.data), d.syg_features_ragged_f32(*args, out.ctypes.data, None),
               d.syg_segment_vectors_ragged_host_f32(*args, ids, out.ctypes.data)):
        assert rc == _ffi.SYG_E_UNSUPPORTED
        assert eng.lib.last_feature_frames() == 0
    assert (out == 7.0).all()
    with pytest.raises(NotImplementedError):
        eng.lib.ragged_frame_offsets(units, 512, 160)
    ok = eng.ragged_units([4], [G31 - 1], len(y))                    # one sample less is a valid unit
    assert eng.lib.ragged_frame_offsets(ok, 512, 160)[-1] == eng.frame_count(G31 - 1, 512, 160)


# ------------------------------------------------------------------------------------------------ PCM ingest
def test_pcm_s16_stereo_past_2g_frames(eng):
    """syg_features_host_pcm / syg_segment_vectors_host_pcm on an s16 stereo payload with units past frame 2^31 (byte 2^33):
    bit-equal to the float32 path on the same (de-interleaved, averaged, widened) samples."""
    sr, fl, hop = 22050, 1024, 256
    feats, fp = ["mfcc", "spectral_centroid", "rms_energy", "crest_factor"], {"mfcc": {"n_mels": 40}}
    L = 4000
    n = G31 + REGION
    raw = np.zeros((n, 2), np.int16)
    mono = np.zeros(n, np.float32)
    rng = np.random.default_rng(3)
    for lo, hi in ((G31 - REGION, n),):
        pcm = np.clip(rng.standard_normal((hi - lo, 2)) * 6000, -32768, 32767).astype(np.int16)
        raw[lo:hi] = pcm
        mono[lo:hi] = orc.load_audio_payload(pcm.tobytes(), _ffi.PCM_S16, 2, mono=True)
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    rows = eng.rows(p)
    # the host pipeline copies each chunk's span: every unit sits near frame 2^31
    starts = np.array([G31 - L // 2 - 1, G31 + 7, G31 + 12345, n - L // 3], np.int64)
    valid = np.array([L, L // 2, L, L // 3], np.int32)
    u = eng.units_table(starts.ctypes.data, valid.ctypes.data, len(starts), L, n)
    a = eng.features_host_pcm(raw.ctypes.data, _ffi.PCM_S16, 2, u, p)
    b = eng.features_host(mono, u, p)
    assert np.array_equal(a, b)
    ids = [r % len(AGG) for r in range(rows)]
    va = eng.segment_vectors_host(raw.ctypes.data, u, p, ids, fmt=_ffi.PCM_S16, channels=2)
    vb = eng.segment_vectors_host(mono.ctypes.data, u, p, ids)
    assert np.array_equal(va, vb)
    names = batch.feature_row_names(feats, fp)
    _, ref = oracle_rows(unit_window(mono, int(starts[2]), L, L), sr, feats, fl, hop, fp)
    check_rows(names, a[2], ref, bin_hz=sr / fl, nyq=sr / 2)


# ------------------------------------------------------------------------------------------------ aggregation
def test_aggregate_offsets_and_row_stride_past_2g(eng):
    """syg_aggregate_f32 with seg_off past 2^31 and row_stride past 2^31 (explicit offsets), and with s * n_rows * row_stride past
    2^31 (regular layout): equal to the same segments near 0 and to the oracle's formatter."""
    rows, n = 2, 300
    stride = G31 + 5000
    offs = np.array([3, G31 - 150, G31 + 1011, G31 // 2], np.int64)          # rows never overlap another segment's rows
    lens = np.array([n, n, n - 1, 1], np.int32)
    rng = np.random.default_rng(2)
    big = Lazy(int(offs.max()) + stride + n + 16)
    vals = []
    for o, ln in zip(offs, lens):
        v = rng.standard_normal((rows, ln)).astype(np.float32)
        v[0, ::7] = np.nan
        for r in range(rows):
            big.put(int(o) + r * stride, v[r])
        vals.append(v)
    got = {}
    with device(eng, big) as (pf,):
        hold, (po, pl_) = _dev_buffers(eng, offs, lens)
        for agg in AGG:
            h, (pout,) = _dev_buffers(eng, np.zeros((len(offs), rows)))
            eng.aggregate_dev(pf, len(offs), rows, stride, [AGG.index(agg)] * rows, pout, seg_off_ptr=po, seg_len_ptr=pl_)
            sync(eng)
            got[agg] = _host(eng, h[0])
    # the same segments packed near 0 (offsets keep their value modulo 4)
    small = np.full((rows, 4 * 512), np.nan, np.float32)
    offs2 = np.array([512 * i + int(o) % 4 for i, o in enumerate(offs)], np.int64)
    for o2, v in zip(offs2, vals):
        small[:, o2:o2 + v.shape[1]] = v
    for agg in AGG:
        h2, (pm2, po2, pl2, pout2) = _dev_buffers(eng, small, offs2, lens, np.zeros((len(offs), rows)))
        eng.aggregate_dev(pm2, len(offs), rows, small.shape[1], [AGG.index(agg)] * rows, pout2, seg_off_ptr=po2, seg_len_ptr=pl2)
        sync(eng)
        assert np.array_equal(got[agg], _host(eng, h2[3]), equal_nan=True), agg
        ref = np.array([[orc.format_feature_vectors_per_segment({"x": v[r].astype(np.float64)}, [(0, v.shape[1])], agg)[0][0]
                         for r in range(rows)] for v in vals])
        if agg in ("median", "min", "max"):
            assert np.array_equal(got[agg], ref, equal_nan=True), agg
        else:
            np.testing.assert_allclose(got[agg], ref, rtol=1e-12, atol=1e-12)
    # regular layout: segment s, row r at (s * rows + r) * rs; both rows of segment 1 sit past 2^31
    rs = G31 // 2 + 3
    reg = Lazy(3 * rs + 64)
    cube = rng.standard_normal((2, rows, 40)).astype(np.float32)
    for s in range(2):
        for r in range(rows):
            reg.put((s * rows + r) * rs, cube[s, r])
    ids = [AGG.index("median"), AGG.index("mean")]
    with device(eng, reg) as (pf,):
        hold, (pout,) = _dev_buffers(eng, np.zeros((2, rows)))
        eng.aggregate_dev(pf, 2, rows, rs, ids, pout, fixed_len=40)
        sync(eng)
        got = _host(eng, hold[0])
    ref = np.array([[np.median(cube[s, 0].astype(np.float64)), cube[s, 1].astype(np.float64).mean()] for s in range(2)])
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=0)


# ------------------------------------------------------------------------------------------------ segmentation arithmetic
def segment_formulas(total, sr, sec, ovl, pad, min_sec):
    """segmentation.py:62-114 restated on index arrays (the oracle's loop would build a multi-GB list here)."""
    seg = int(sec * sr)
    hop = max(1, int(seg * (1.0 - ovl)))
    mn = int(min_sec * sr) if min_sec is not None else 0
    starts = np.arange(0, total, hop, dtype=np.int64)
    if not pad:                                    # the loop stops before a start whose segment would pass the end
        starts = starts[(starts == 0) | (starts + seg <= total)]
    orig = np.minimum(starts + seg, total) - starts
    keep = (starts + seg <= total) | pad
    if mn > 0:
        keep &= orig >= mn
    return seg, hop, starts[keep], orig[keep]


@pytest.mark.parametrize("total", [G31 - 1, G31, G32 + 1, 30 * 3600 * 48000])
@pytest.mark.parametrize("sec,ovl,pad,min_sec", [(2.0, 0.5, True, None), (1.0, 0.0, False, None), (3.7, 0.25, True, 1.0)])
def test_segment_table_large_totals(total, sec, ovl, pad, min_sec):
    sr = 48000
    seg, hop, st, va = _ffi.library().segment_table(total, sr, sec, ovl, pad, min_sec)
    rseg, rhop, rst, rva = segment_formulas(total, sr, sec, ovl, pad, min_sec)
    assert (seg, hop, len(st)) == (rseg, rhop, len(rst))
    assert st[0] == rst[0] and st[-1] == rst[-1] and va[-1] == rva[-1]
    assert np.array_equal(st, rst) and np.array_equal(va, rva)
    assert st[-1] < total and st[-1] + va[-1] <= total


# ------------------------------------------------------------------------------------------------ outputs past 2^31 elements
def long_input(n, sr, seed):
    """n samples on the device: a 2^20-sample mixture repeated (a unit's content is what matters, not its uniqueness)"""
    import torch
    return torch.from_numpy(synth.mixture(1 << 20, sr, seed=seed)).cuda().repeat(n // (1 << 20) + 1)[:n].contiguous()


def last_units_equal(eng, run_one, full, n_units, k=3):
    """the last k units of a big launch == the same units in a launch of their own"""
    for u in range(n_units - k, n_units):
        assert np.array_equal(run_one(u), full(u), equal_nan=True), f"unit {u}"


@pytest.mark.gpu
def test_stft_power_output_past_2g():
    """stft_dev power output of 256k overlapping units: the last units' outputs sit past element 2^31 (ring kernel)."""
    import torch
    eng = get_engine("gpu")
    n_fft, hop, L, stride = 256, 64, 4096, 256
    B, T = 1 + n_fft // 2, eng.frame_count(L, n_fft, hop)
    n_units = G31 // (B * T) + 64
    total = (n_units - 1) * stride + L
    assert (n_units - 1) * B * T > G31
    need_device_bytes(n_units * B * T * 4 + total * 4)
    y = long_input(total, 22050, seed=4)
    out = torch.empty((n_units, B, T), dtype=torch.float32, device="cuda")
    try:
        eng.stft_dev(y.data_ptr(), eng.units_clips(n_units, L, total_len=total, stride=stride), n_fft, hop, n_fft, 0, True, 0,
                     _ffi.OUT_POWER, out.data_ptr())
        torch.cuda.synchronize()
        path = eng.lib.dll.syg_debug_last_stft_path()
        assert path == 1
        one = torch.empty((1, B, T), dtype=torch.float32, device="cuda")

        def single(u):
            eng.stft_dev(y.data_ptr() + 4 * u * stride, eng.units_clips(1, L, total_len=total - u * stride), n_fft, hop, n_fft, 0,
                         True, 0, _ffi.OUT_POWER, one.data_ptr())
            torch.cuda.synchronize()
            assert eng.lib.dll.syg_debug_last_stft_path() == path
            return one[0].cpu().numpy()

        last_units_equal(eng, single, lambda u: out[u].cpu().numpy(), n_units)
        u = n_units - 1
        seg = y[u * stride:u * stride + L].cpu().numpy().astype(np.float64)
        power_close(out[u].cpu().numpy().astype(np.float64), np.abs(orc.compute_stft(seg, n_fft=n_fft, hop_length=hop)) ** 2)
    finally:
        del y, out
        torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("feats", [["mfcc", "rms_energy"], ["mfcc", "spectral_contrast", "rms_energy", "spectral_centroid"]])
def test_features_dev_output_past_2g(feats):
    """features_dev with n_units x n_rows x T > 2^31 on the resident epilogue (MFCC only) and the two-kernel path (contrast)."""
    import torch
    eng = get_engine("gpu")
    sr, fl, hop, L, stride = 16000, 512, 160, 16000, 160
    fp = {"mfcc": {"n_mels": 40}}
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    rows, T = eng.rows(p), eng.frame_count(L, fl, hop)
    n_units = G31 // (rows * T) + 64
    total = (n_units - 1) * stride + L
    need_device_bytes(n_units * rows * T * 4 + total * 4 + (2 << 30))
    y = long_input(total, sr, seed=6)
    out = torch.empty((n_units, rows, T), dtype=torch.float32, device="cuda")
    resident_path = len(feats) == 2
    try:
        eng.features_dev(y.data_ptr(), eng.units_clips(n_units, L, total_len=total, stride=stride), p, out.data_ptr())
        torch.cuda.synchronize()
        assert eng.lib.dll.syg_debug_last_features_resident() == int(resident_path)
        one = torch.empty((1, rows, T), dtype=torch.float32, device="cuda")

        def single(u):
            with resident(eng, resident_path):
                eng.features_dev(y.data_ptr() + 4 * u * stride, eng.units_clips(1, L), p, one.data_ptr())
                torch.cuda.synchronize()
                assert eng.lib.dll.syg_debug_last_features_resident() == int(resident_path)
            return one[0].cpu().numpy()

        last_units_equal(eng, single, lambda u: out[u].cpu().numpy(), n_units)
        u = n_units - 1
        names, ref = oracle_rows(y[u * stride:u * stride + L].cpu().numpy(), sr, feats, fl, hop, fp)
        check_rows(names, out[u].cpu().numpy(), ref, bin_hz=sr / fl, nyq=sr / 2)
    finally:
        del y, out
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_features_ragged_dev_output_past_2g():
    """features_ragged_dev with n_rows x F > 2^31: overlapping units of their own lengths; the last units' columns of the last
    rows sit past element 2^31."""
    import torch
    eng = get_engine("gpu")
    sr, fl, hop, feats, fp = RAGGED
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    rows = eng.rows(p)
    rng = np.random.default_rng(8)
    n_units = G31 // (rows * 100) + 1000
    lengths = rng.integers(14000, 18000, n_units).astype(np.int64)
    starts = np.arange(n_units, dtype=np.int64) * 160
    total = int((starts + lengths).max())
    units = eng.ragged_units(starts, lengths, total)
    foff = eng.lib.ragged_frame_offsets(units, fl, hop)
    F = int(foff[-1])
    assert rows * F > G31
    need_device_bytes(rows * F * 4 + total * 4 + (2 << 30))
    y = long_input(total, sr, seed=9)
    out = torch.empty((rows, F), dtype=torch.float32, device="cuda")
    try:
        eng.features_ragged_dev(y.data_ptr(), units, p, out.data_ptr())
        torch.cuda.synchronize()
        assert eng.lib.last_feature_frames() == F

        def single(u):
            uu = eng.ragged_units([int(starts[u])], [int(lengths[u])], total)
            o = torch.empty((rows, int(foff[u + 1] - foff[u])), dtype=torch.float32, device="cuda")
            eng.features_ragged_dev(y.data_ptr(), uu, p, o.data_ptr())
            return o.cpu().numpy()

        last_units_equal(eng, single, lambda u: out[:, int(foff[u]):int(foff[u + 1])].cpu().numpy(), n_units)
        u = n_units - 1
        names, ref = oracle_rows(y[int(starts[u]):int(starts[u] + lengths[u])].cpu().numpy(), sr, feats, fl, hop, fp)
        check_rows(names, out[:, int(foff[u]):int(foff[u + 1])].cpu().numpy(), ref, bin_hz=sr / fl, nyq=sr / 2)
    finally:
        del y, out
        torch.cuda.empty_cache()
