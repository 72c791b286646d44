"""Ragged batches: units of their own lengths in one call (syg_*_ragged_*, batch.extract_features_ragged / clip_vectors).

The contract: unit u is exactly y[starts[u], starts[u] + lengths[u]); its T_u frames sit at columns F_u .. F_{u+1}-1 of the
[n_rows][F] output and equal, bit for bit, what the uniform entry points return for that unit alone (its own power_to_db reference
level included).  Each case also matches the float64 oracle at the tolerances of test_parity_cabi.py, and the segment vectors
equal syg_aggregate_f32 on the ragged block and the oracle's format_feature_vectors_per_segment."""
import numpy as np
import pytest

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi, batch
from sygnals_b200.utils import synth
from test_parity_cabi import _dev_buffers, _host, check_rows, oracle_rows

ALL16 = list(_ffi.FEATURE_IDS)
CFG4 = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]

# name -> (sr, frame_length, hop, features, feature_params, base length of the ordinary units)
CASES = {
    "warp512": (16000, 512, 160, ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"],
                {"mfcc": {"n_mels": 40}}, 700),
    "spec44kl": (44100, 2048, 512, CFG4, None, 1000),
    "all16_2048": (44100, 2048, 512, ALL16, None, 1000),
    "spec22k": (22050, 2048, 512, ["mfcc", "rms_energy"], {"mfcc": {"n_mels": 128, "n_mfcc": 20}}, 1000),
    "block4096": (48000, 4096, 1024, ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy",
                                      "zero_crossing_rate"], None, 2000),
    "mixed1000": (16000, 1000, 250, ["mfcc", "spectral_centroid", "spectral_rolloff", "rms_energy", "skewness"], {"mfcc": {"n_mels": 40}}, 900),
    "mixed441": (22050, 441, 147, ["mfcc", "spectral_contrast", "rms_energy", "peak_amplitude"], {"mfcc": {"n_mels": 40}}, 800),
}


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


def ragged_batch(fl, hop, base, seed, center=True):
    """(y, starts, lengths, scales): lengths 0, 1, hop - 1, fl - 1, exact hop multiples, ordinary ones and one 50x longer unit;
    a silent unit, units scaled by 1e-3 / 1e-6, gaps between units and two windows overlapping their neighbours."""
    rng = np.random.default_rng(seed)
    lengths = [0, 1, hop - 1, fl - 1, 2 * hop, 5 * hop, base, base + 37, 50 * base, base // 2 + 3, base, base, 3 * hop + 1]
    scales = [1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0.0, 1e-3, 1e-6]
    if not center:
        lengths += [fl // 2, fl - 1, 0]       # no frames without centring
        scales += [1, 1, 1]
    pieces, starts, pos = [], [], 0
    for i, (n, s) in enumerate(zip(lengths, scales)):
        gap = int(rng.integers(0, 7))
        pieces.append(np.zeros(gap, np.float32))
        pos += gap
        starts.append(pos)
        pieces.append((synth.mixture(n, 16000, seed=seed + i) * np.float32(s)).astype(np.float32) if n else np.zeros(0, np.float32))
        pos += n
    y = np.concatenate(pieces)
    # overlapping windows: the second half of the long unit into the next one, and a window inside an ordinary unit
    starts += [starts[8] + 25 * base, starts[6] + 11]
    lengths += [25 * base + lengths[9] + 3, base // 3]
    assert starts[-2] + lengths[-2] <= len(y)
    return y, np.array(starts, np.int64), np.array(lengths, np.int64)


def params(eng, case, center=True):
    sr, fl, hop, feats, fp, _ = CASES[case]
    return _ffi.make_params(eng.lib, sr, feats, fl, hop, center=center, feature_params=fp)


@pytest.mark.parametrize("case", list(CASES))
def test_ragged_equals_single_units_and_oracle(eng, case):
    sr, fl, hop, feats, fp, base = CASES[case]
    y, starts, lengths = ragged_batch(fl, hop, base, seed=len(case))
    p = params(eng, case)
    units = eng.ragged_units(starts, lengths, len(y))
    foff = eng.lib.ragged_frame_offsets(units, fl, hop, True)
    assert list(np.diff(foff)) == [eng.frame_count(int(n), fl, hop, True) for n in lengths]
    if fl % 2 == 0:                                    # manager.py's frame count rule holds for even frame lengths
        assert list(np.diff(foff)) == [orc.frame_count(int(n), fl, hop, True) for n in lengths]
    out = eng.features_ragged_host(y, units, p)
    assert out.shape == (eng.rows(p), foff[-1])
    assert eng.lib.last_feature_frames() == foff[-1]
    assert eng.lib.dll.syg_debug_last_features_resident() == 0
    names = batch.feature_row_names(feats, fp)
    for u, (s, n) in enumerate(zip(starts, lengths)):
        seg = y[s:s + n]
        one = eng.features_host(seg, eng.units_clips(1, int(n)), p)
        got = out[:, foff[u]:foff[u + 1]]
        assert np.array_equal(one[0], got, equal_nan=True), f"unit {u} (length {n}) differs from its single-unit result"
        if n > 0 and np.abs(seg).max() >= 1e-4:
            ref_names, ref = oracle_rows(seg, sr, feats, fl, hop, feature_params=fp)
            assert ref_names == names
            check_rows(names, got, ref, bin_hz=sr / fl, nyq=sr / 2)


@pytest.mark.parametrize("case", ["warp512", "mixed1000"])
def test_ragged_uncentred_zero_frame_units(eng, case):
    sr, fl, hop, feats, fp, base = CASES[case]
    y, starts, lengths = ragged_batch(fl, hop, base, seed=3, center=False)
    p = params(eng, case, center=False)
    units = eng.ragged_units(starts, lengths, len(y))
    foff = eng.lib.ragged_frame_offsets(units, fl, hop, False)
    T = np.diff(foff)
    assert list(T) == [orc.frame_count(int(n), fl, hop, False) for n in lengths]
    assert (T == 0).sum() >= 4
    out = eng.features_ragged_host(y, units, p)
    assert eng.lib.last_feature_frames() == foff[-1]
    for u, (s, n) in enumerate(zip(starts, lengths)):
        one = eng.features_host(y[s:s + n], eng.units_clips(1, int(n)), p)
        assert np.array_equal(one[0], out[:, foff[u]:foff[u + 1]], equal_nan=True), f"unit {u}"
    # segment vectors: zero-frame units are the reference's skipped segments (NaN rows)
    vec = eng.segment_vectors_ragged_host(y, units, p, [0] * eng.rows(p))
    assert np.isnan(vec[T == 0]).all() and not np.isnan(vec[T > 0]).any()


@pytest.mark.parametrize("agg", ["mean", "std", "median", "min", "max", "mixed"])
def test_ragged_segment_vectors(eng, agg):
    case = "warp512"
    sr, fl, hop, feats, fp, base = CASES[case]
    y, starts, lengths = ragged_batch(fl, hop, base, seed=21)
    p = params(eng, case)
    names = batch.feature_row_names(feats, fp)
    aggregation = {"mfcc_0": "median", "mfcc_3": "std", "spectral_centroid": "max", "rms_energy": "min"} if agg == "mixed" else agg
    ids = [_ffi.AGG_IDS[aggregation.get(n, "mean") if isinstance(aggregation, dict) else aggregation] for n in names]
    units = eng.ragged_units(starts, lengths, len(y))
    foff = eng.lib.ragged_frame_offsets(units, fl, hop, True)
    vec = eng.segment_vectors_ragged_host(y, units, p, ids)
    assert eng.lib.last_feature_frames() == foff[-1]
    feats_rows = eng.features_ragged_host(y, units, p)
    # == syg_aggregate_f32 on the ragged block with offsets F_u and lengths T_u, bit for bit
    off = foff[:-1].astype(np.int64)
    ln = np.diff(foff).astype(np.int32)
    ref_out = np.zeros_like(vec)
    hold, (pm, po, pl_, pout) = _dev_buffers(eng, feats_rows, off, ln, ref_out)
    eng.aggregate_dev(pm, len(lengths), len(names), foff[-1], ids, pout, seg_off_ptr=po, seg_len_ptr=pl_)
    if not isinstance(hold[3], np.ndarray):
        import torch
        torch.cuda.synchronize()
    assert np.array_equal(vec, _host(eng, hold[3]), equal_nan=True)
    # == the oracle's format_feature_vectors_per_segment on the engine's own per-unit rows
    d = {n: feats_rows[r].astype(np.float64) for r, n in enumerate(names)}
    ref = orc.format_feature_vectors_per_segment(d, [(int(foff[u]), int(foff[u + 1])) for u in range(len(lengths))], aggregation)
    assert np.array_equal(np.isnan(vec), np.isnan(ref))
    ok = ~np.isnan(ref)
    if agg in ("median", "min", "max"):
        assert np.array_equal(vec[ok], ref[ok])
    else:
        np.testing.assert_allclose(vec[ok], ref[ok], rtol=1e-12, atol=1e-12)


def test_ragged_device_form_and_chunks(eng):
    """Host and device forms agree; a 1 MiB workspace cuts the batch into several chunks, one unit bigger than the limit runs
    alone, and nothing changes."""
    sr, fl, hop = 16000, 512, 16
    feats, fp = ["mfcc", "spectral_contrast", "rms_energy"], {"mfcc": {"n_mels": 64}}
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, feature_params=fp)
    lengths = np.array([3000, 60000, 0, 5000, 8000, 4100, 2500, 7000, 6000, 511, 9000], np.int64)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    y = synth.mixture(int(lengths.sum()), sr, seed=8)
    units = eng.ragged_units(starts, lengths, len(y))
    foff = eng.lib.ragged_frame_offsets(units, fl, hop, True)
    rows = eng.rows(p)
    ids = [_ffi.AGG_IDS["mean"]] * rows
    ref_f = eng.features_ragged_host(y, units, p)
    ref_v = eng.segment_vectors_ragged_host(y, units, p, ids)
    assert int(np.diff(foff).max()) * (64 + 14 + 2) * 4 > (1 << 20)       # the long unit alone exceeds the workspace limit
    try:
        eng.set_workspace_limit(1 << 20)
        f_small = eng.features_ragged_host(y, units, p)
        v_small = eng.segment_vectors_ragged_host(y, units, p, ids)
        out_f = np.zeros((rows, foff[-1]), np.float32)
        out_v = np.zeros((len(lengths), rows), np.float64)
        hold, (py, pf, pv) = _dev_buffers(eng, y, out_f, out_v)
        eng.features_ragged_dev(py, units, p, pf)
        assert eng.lib.last_feature_frames() == foff[-1]
        eng.segment_vectors_ragged_dev(py, units, p, ids, pv)
        if not isinstance(hold[0], np.ndarray):
            import torch
            torch.cuda.synchronize()
        d_f, d_v = _host(eng, hold[1]), _host(eng, hold[2])
    finally:
        eng.set_workspace_limit(1 << 30)
    for got in (f_small, d_f):
        assert np.array_equal(got, ref_f, equal_nan=True)
    for got in (v_small, d_v):
        assert np.array_equal(got, ref_v, equal_nan=True)


@pytest.mark.parametrize("lengths,hop,ws", [([300, 5000], 160, None), ([60000, 300, 400, 60000], 16, 1 << 20)])
def test_ragged_chunk_without_frames(eng, lengths, hop, ws):
    """Chunks that hold only units without frames (center=False, length < frame_length): the host forms' two-lane split puts the
    300-sample clip of [300, 5000] in a chunk of its own; a 1 MiB workspace cuts [60000, 300, 400, 60000] (hop 16) into
    {60000}, {300, 400}, {60000} in the device form too.  Nothing is launched for such a chunk; its vectors are NaN rows."""
    sr, fl = 16000, 512
    feats, fp = ["mfcc", "spectral_contrast", "rms_energy"], {"mfcc": {"n_mels": 64}}
    p = _ffi.make_params(eng.lib, sr, feats, fl, hop, center=False, feature_params=fp)
    lengths = np.array(lengths, np.int64)
    starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    y = synth.mixture(int(lengths.sum()), sr, seed=31)
    units = eng.ragged_units(starts, lengths, len(y))
    foff = eng.lib.ragged_frame_offsets(units, fl, hop, False)
    T = np.diff(foff)
    assert (T == 0).any() and foff[-1] > 0
    rows = eng.rows(p)
    ids = [_ffi.AGG_IDS["mean"]] * rows
    singles = [eng.features_host(y[s:s + n], eng.units_clips(1, int(n)), p)[0] for s, n in zip(starts, lengths)]
    try:
        if ws:
            eng.set_workspace_limit(ws)
        h_f = eng.features_ragged_host(y, units, p)
        assert eng.lib.last_feature_frames() == foff[-1]
        h_v = eng.segment_vectors_ragged_host(y, units, p, ids)
        out_f = np.zeros((rows, foff[-1]), np.float32)
        out_v = np.zeros((len(lengths), rows), np.float64)
        hold, (py, pf, pv) = _dev_buffers(eng, y, out_f, out_v)
        eng.features_ragged_dev(py, units, p, pf)
        assert eng.lib.last_feature_frames() == foff[-1]
        eng.segment_vectors_ragged_dev(py, units, p, ids, pv)
        if not isinstance(hold[0], np.ndarray):
            import torch
            torch.cuda.synchronize()
        d_f, d_v = _host(eng, hold[1]), _host(eng, hold[2])
    finally:
        eng.set_workspace_limit(1 << 30)
    for f in (h_f, d_f):
        for u in range(len(lengths)):
            assert np.array_equal(f[:, foff[u]:foff[u + 1]], singles[u], equal_nan=True), f"unit {u}"
    for v in (h_v, d_v):
        assert np.isnan(v[T == 0]).all()
        for u in np.flatnonzero(T):
            np.testing.assert_allclose(v[u], singles[u].astype(np.float64).mean(axis=1), rtol=1e-12, atol=1e-12)


def test_ragged_errors(eng):
    p = _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160)
    y = np.zeros(4000, np.float32)
    with pytest.raises(ValueError, match="negative"):
        eng.features_ragged_host(y, eng.ragged_units([0, 10], [100, -1], len(y)), p)
    with pytest.raises(ValueError, match="outside"):
        eng.features_ragged_host(y, eng.ragged_units([0, 3900], [100, 101], len(y)), p)
    with pytest.raises(ValueError, match="negative"):
        eng.lib.ragged_frame_offsets(eng.ragged_units([-1], [10], len(y)), 512, 160)
    null = _ffi.SygRaggedUnits(2, len(y), None, None)
    with pytest.raises(ValueError, match="NULL"):
        eng.features_ragged_host(y, null, p)
    with pytest.raises(ValueError, match="NULL"):
        eng.segment_vectors_ragged_host(y, null, p, [0] * 13)
    with pytest.raises(NotImplementedError):                                   # 2 * 503: no kernel for this length
        eng.features_ragged_host(y, eng.ragged_units([0], [4000], len(y)), _ffi.make_params(eng.lib, 16000, ["mfcc"], 1006, 160))
    with pytest.raises(NotImplementedError):                                   # a unit longer than 2^31-1 samples
        eng.lib.ragged_frame_offsets(eng.ragged_units([0], [1 << 31], 1 << 32), 512, 160)
    # nothing to do: no units, or no frames at all
    empty = eng.features_ragged_host(y, eng.ragged_units([], [], len(y)), p)
    assert empty.shape == (13, 0)
    p_nc = _ffi.make_params(eng.lib, 16000, ["mfcc"], 512, 160, center=False)
    none = eng.features_ragged_host(y, eng.ragged_units([0, 5], [100, 511], len(y)), p_nc)
    assert none.shape == (13, 0) and eng.lib.last_feature_frames() == 0


def test_ragged_input_forms():
    """The forms of ``clips`` resolve to the same (y, starts, lengths) (no device needed)."""
    clips = [synth.mixture(n, 16000, seed=n) for n in (300, 0, 1000, 17)]
    y, st, ln = batch._ragged_input(clips)
    assert list(ln) == [300, 0, 1000, 17] and list(st) == [0, 300, 300, 1300]
    assert np.array_equal(y, np.concatenate(clips), equal_nan=True)
    y2, st2, ln2 = batch._ragged_input(batch.Windows(y, st, list(ln)))
    assert y2 is y and np.array_equal(st2, st) and np.array_equal(ln2, ln)
    # a plain tuple is always a sequence of clips, whatever their dtype: no guessing between clips and a window table
    y3, st3, ln3 = batch._ragged_input(tuple(clips[:3]))
    assert list(ln3) == [300, 0, 1000] and len(y3) == 1300
    pcm = tuple(np.arange(n, dtype=np.int16) for n in (5, 3, 4))
    y4, st4, ln4 = batch._ragged_input(pcm)
    assert list(ln4) == [5, 3, 4] and y4.dtype == np.float32 and len(y4) == 12
    with pytest.raises(ValueError):
        batch._ragged_input([np.zeros((2, 3), np.float32)])
    with pytest.raises(ValueError):
        batch._ragged_input(batch.Windows(y, st, ln[:2]))
    with pytest.raises(ValueError):
        batch._ragged_input(batch.Windows(y, st.astype(np.float64), ln))


@pytest.mark.gpu
def test_python_functions_all_forms():
    import torch
    sr, fl, hop = 44100, 2048, 512
    lengths = [int(x) for x in np.random.default_rng(5).integers(1000, 30000, 9)] + [0, 511]
    clips = [synth.mixture(n, sr, seed=i) for i, n in enumerate(lengths)]
    eng = _ffi.engine(0)
    p = _ffi.make_params(eng.lib, sr, CFG4, fl, hop)
    y = np.concatenate(clips)
    st = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
    units = eng.ragged_units(st, lengths, len(y))
    ref_f = eng.features_ragged_host(y, units, p)
    ids = [_ffi.AGG_IDS["median"]] * eng.rows(p)
    ref_v = eng.segment_vectors_ragged_host(y, units, p, ids)
    yd = torch.from_numpy(y).cuda()
    forms = [clips, batch.Windows(y, st, lengths), [torch.from_numpy(c).cuda() for c in clips],
             batch.Windows(yd, torch.from_numpy(st).cuda(), torch.tensor(lengths).cuda())]
    for form in forms:
        r = batch.extract_features_ragged(form, sr, CFG4, fl, hop)
        names, v = batch.clip_vectors(form, sr, CFG4, aggregation="median", frame_length=fl, hop_length=hop)
        f = r["features"].cpu().numpy() if torch.is_tensor(r["features"]) else r["features"]
        v = v.cpu().numpy() if torch.is_tensor(v) else v
        assert r["names"] == names == batch.feature_row_names(CFG4)
        assert np.array_equal(r["frame_offsets"], eng.lib.ragged_frame_offsets(units, fl, hop))
        assert np.array_equal(f, ref_f, equal_nan=True)
        assert np.array_equal(v, ref_v, equal_nan=True)
    # per-feature dict as formatters._agg_ids takes it
    agg = {"mfcc_0": "max", "spectral_rolloff": "std"}
    names, v = batch.clip_vectors(clips, sr, CFG4, aggregation=agg, frame_length=fl, hop_length=hop)
    ids = [_ffi.AGG_IDS[agg.get(n, "mean")] for n in names]
    assert np.array_equal(v, eng.segment_vectors_ragged_host(y, units, p, ids), equal_nan=True)
