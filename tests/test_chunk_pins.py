"""Where each chunked entry point cuts its units into chunks, pinned.

Results do not depend on the cut, so the bit-equality tests cannot see a changed one; but the cut decides which kernels run (the
unit-resident epilogue needs `min_groups` unit groups in its chunk) and how many launches a call issues.  Every call here runs under
a 1 MiB workspace limit and under the default one, with the resident minimum lowered so that the last chunks of the two limits
choose differently.  After each call the debug getters, which describe the call's last chunk (frames of the call, finalize tile
height / CTAs / tiles, resident epilogue, mel projection form), and on the B200 the launches per kind, must equal the literal
values below; the outputs of the two limits must be equal bit for bit."""
import numpy as np
import pytest

from backends import BACKENDS, get_engine
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth
from test_parity_cabi import _dev_buffers, _host

SMALL, DEFAULT = 1 << 20, 1 << 30
MIN_GROUPS = 6            # the default limit's last chunks have at least 6 unit groups, the 1 MiB limit's last chunks fewer

SR, FL, HOP = 16000, 256, 64
# device forms: 40 frames and 20 KB of mel energies per unit, 51 units per chunk under 1 MiB; 3 units per resident group
N_DEV, L_DEV, T_DEV, STRIDE_DEV, FP_DEV = 56, 39 * HOP, 40, 2000, {"mfcc": {"n_mels": 128}}
# host forms, which split their units between two lanes first: one frame and 768 bytes of workspace per unit (three parts aligned
# to 256 bytes and 256 spare), so 1365 units per chunk under 1 MiB; 256 units per resident group
N_HOST, L_HOST, STRIDE_HOST, FP_HOST = 2800, HOP - 1, 50, {"mfcc": {"n_mels": 32, "n_mfcc": 2}}


def _clips(n, unit_len, stride, seed):
    y = synth.mixture((n - 1) * stride + unit_len, SR, seed=seed)
    return y, (n, unit_len, len(y), stride)


def _tables(n, unit_len, seed):
    """Explicit unit tables: starts with gaps, every fifth unit shorter than unit_len (its frames read zeros past its end)."""
    rng = np.random.default_rng(seed)
    starts = np.cumsum(rng.integers(unit_len // 2, unit_len * 3 // 2, n)).astype(np.int64)
    valid = np.where(np.arange(n) % 5 == 2, unit_len // 3, unit_len).astype(np.int32)
    return starts, valid, int(starts[-1]) + unit_len


def _ragged_batch(n):
    """n units of 0 to 3999 samples (some without frames: the ragged calls do not centre), gaps between them."""
    rng = np.random.default_rng(n)
    lengths = rng.integers(0, 4000, n).astype(np.int64)
    lengths[[3, 17]] = [0, 40]
    starts = np.cumsum(np.concatenate([[5], lengths[:-1] + rng.integers(0, 9, n - 1)])).astype(np.int64)
    return synth.mixture(int(starts[-1] + lengths[-1]) + 3, SR, seed=n + 1), starts, lengths


def _ragged_params(eng):
    return _ffi.make_params(eng.lib, SR, ["mfcc", "spectral_contrast", "rms_energy"], FL, HOP, center=False,
                            feature_params={"mfcc": {"n_mels": 256}})


def _dev_params(eng):
    return _ffi.make_params(eng.lib, SR, ["mfcc", "rms_energy", "zero_crossing_rate"], FL, HOP, feature_params=FP_DEV)


def _host_params(eng):
    return _ffi.make_params(eng.lib, SR, ["mfcc", "rms_energy"], FL, HOP, feature_params=FP_HOST)


def _agg_ids(eng, p):
    return [(0, 1, 3, 4)[i % 4] for i in range(eng.rows(p))]        # mean, std, min, max (medians are slow to emulate)


def _sync(hold):
    if not isinstance(hold[0], np.ndarray):
        import torch
        torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- the calls
def features_dev_stride(eng):
    p = _dev_params(eng)
    y, (n, unit_len, total, stride) = _clips(N_DEV, L_DEV, STRIDE_DEV, 1)
    hold, (py, po) = _dev_buffers(eng, y, np.zeros((n, eng.rows(p), T_DEV), np.float32))
    eng.features_dev(py, eng.units_clips(n, unit_len, total, stride), p, po)
    _sync(hold)
    return _host(eng, hold[1])


def features_dev_tables(eng):
    p = _dev_params(eng)
    starts, valid, total = _tables(N_DEV, L_DEV, 2)
    y = synth.mixture(total, SR, seed=3)
    hold, (py, ps, pv, po) = _dev_buffers(eng, y, starts, valid, np.zeros((N_DEV, eng.rows(p), T_DEV), np.float32))
    eng.features_dev(py, eng.units_table(ps, pv, N_DEV, L_DEV, total), p, po)
    _sync(hold)
    return _host(eng, hold[3])


def segment_vectors_dev(eng):
    p = _dev_params(eng)
    y, (n, unit_len, total, stride) = _clips(N_DEV, L_DEV, STRIDE_DEV, 4)
    hold, (py, po) = _dev_buffers(eng, y, np.zeros((n, eng.rows(p)), np.float64))
    eng.segment_vectors_dev(py, eng.units_clips(n, unit_len, total, stride), p, _agg_ids(eng, p), po)
    _sync(hold)
    return _host(eng, hold[1])


def _pcm_stereo(total, seed):
    two = np.stack([synth.mixture(total, SR, seed=seed), synth.mixture(total, SR, seed=seed + 1)], axis=1)
    return np.ascontiguousarray(np.round(two * 16000.0).astype(np.int16))


def features_host(eng):
    y, (n, unit_len, total, stride) = _clips(N_HOST, L_HOST, STRIDE_HOST, 5)
    return eng.features_host(y, eng.units_clips(n, unit_len, total, stride), _host_params(eng))


def features_host_pcm(eng):
    starts, valid, total = _tables(N_HOST, L_HOST, 6)
    raw = _pcm_stereo(total, 7)
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, N_HOST, L_HOST, total)
    return eng.features_host_pcm(raw.ctypes.data, _ffi.PCM_S16, 2, units, _host_params(eng))


def segment_vectors_host(eng):
    p = _host_params(eng)
    y, (n, unit_len, total, stride) = _clips(N_HOST, L_HOST, STRIDE_HOST, 9)
    return eng.segment_vectors_host(y.ctypes.data, eng.units_clips(n, unit_len, total, stride), p, _agg_ids(eng, p))


def segment_vectors_host_pcm(eng):
    p = _host_params(eng)
    starts, valid, total = _tables(N_HOST, L_HOST, 10)
    raw = _pcm_stereo(total, 11)
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, N_HOST, L_HOST, total)
    return eng.segment_vectors_host(raw.ctypes.data, units, p, _agg_ids(eng, p), fmt=_ffi.PCM_S16, channels=2)


# 1.1 KB of workspace per frame: about 950 frames per chunk under 1 MiB; the host forms also cut at half the frames
# (1068 frames for 39 units, 2086 for 66)
N_RAGGED_DEV, N_RAGGED_HOST = 39, 66


def features_ragged_host(eng):
    y, starts, lengths = _ragged_batch(N_RAGGED_HOST)
    return eng.features_ragged_host(y, eng.ragged_units(starts, lengths, len(y)), _ragged_params(eng))


def segment_vectors_ragged_host(eng):
    y, starts, lengths = _ragged_batch(N_RAGGED_HOST)
    p = _ragged_params(eng)
    return eng.segment_vectors_ragged_host(y, eng.ragged_units(starts, lengths, len(y)), p, _agg_ids(eng, p))


def features_ragged_dev(eng):
    y, starts, lengths = _ragged_batch(N_RAGGED_DEV)
    p = _ragged_params(eng)
    units = eng.ragged_units(starts, lengths, len(y))
    F = int(eng.lib.ragged_frame_offsets(units, FL, HOP, False)[-1])
    hold, (py, po) = _dev_buffers(eng, y, np.zeros((eng.rows(p), F), np.float32))
    eng.features_ragged_dev(py, units, p, po)
    _sync(hold)
    return _host(eng, hold[1])


def segment_vectors_ragged_dev(eng):
    y, starts, lengths = _ragged_batch(N_RAGGED_DEV)
    p = _ragged_params(eng)
    hold, (py, po) = _dev_buffers(eng, y, np.zeros((len(lengths), eng.rows(p)), np.float64))
    eng.segment_vectors_ragged_dev(py, eng.ragged_units(starts, lengths, len(y)), p, _agg_ids(eng, p), po)
    _sync(hold)
    return _host(eng, hold[1])


def stft_host_tables(eng):
    starts, valid, total = _tables(12, 3000, 12)
    y = synth.mixture(total, SR, seed=13)
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, 12, 3000, total)
    return eng.stft_host(y, units, 512, 128, 400, out_kind=_ffi.OUT_MAGNITUDE)


def psd_welch_host_tables(eng):
    starts, valid, total = _tables(12, 3000, 14)
    y = synth.mixture(total, SR, seed=15)
    units = eng.units_table(starts.ctypes.data, valid.ctypes.data, 12, 3000, total)
    psd, stats = eng.psd_welch_host(y, units, SR, 0, 256, 128, 256, stats=True)
    return np.concatenate([psd, stats], axis=1)


def spectral_contrast_from_mag(eng):
    S = np.abs(np.random.default_rng(16).standard_normal((129, 300))).astype(np.float32)
    hold, (ps, po) = _dev_buffers(eng, S, np.zeros((7, 300), np.float32))
    eng.spectral_contrast_from_mag_dev(ps, 129, 300, SR, 6, 200.0, 0.02, po)
    _sync(hold)
    return _host(eng, hold[1])


# ---------------------------------------------------------------------------------------------- pinned values
# call: (pins under 1 MiB, pins under the default limit).  Pins of a feature call: (frames of the call, (finalize tile frames, CTAs,
# tiles), resident epilogue, interval-form mel projection, launches (frame, finalize, welch, other) on the B200); of the other calls:
# (launches,).  Where every chunk of the default limit is resident, the finalize getter still reports the 1 MiB call's last chunk.
PINS = {
    # 1 MiB: 51 units (resident) + 5; default: 56 units (resident)
    features_dev_stride: ((2240, (32, 7, 7), 0, 1, (4, 1, 0, 0)), (2240, (32, 7, 7), 1, 1, (2, 0, 0, 0))),
    features_dev_tables: ((2240, (32, 7, 7), 0, 1, (4, 1, 0, 0)), (2240, (32, 7, 7), 1, 1, (2, 0, 0, 0))),
    # 1 MiB: 45 units (resident) + 11, the frame features share the workspace; default: 56 units (resident)
    segment_vectors_dev: ((2240, (32, 14, 14), 0, 1, (4, 1, 0, 2)), (2240, (32, 14, 14), 1, 1, (2, 0, 0, 1))),
    # 1 MiB: 1365 + 1365 units (resident) + 70; default: 1400 + 1400 (resident); the PCM forms ingest each chunk
    features_host: ((2800, (64, 2, 2), 0, 1, (3, 1, 0, 0)), (2800, (64, 2, 2), 1, 1, (2, 0, 0, 0))),
    features_host_pcm: ((2800, (64, 2, 2), 0, 1, (3, 1, 0, 3)), (2800, (64, 2, 2), 1, 1, (2, 0, 0, 2))),
    segment_vectors_host: ((2800, (64, 2, 2), 0, 1, (3, 1, 0, 3)), (2800, (64, 2, 2), 1, 1, (2, 0, 0, 2))),
    segment_vectors_host_pcm: ((2800, (64, 2, 2), 0, 1, (3, 1, 0, 6)), (2800, (64, 2, 2), 1, 1, (2, 0, 0, 4))),
    # 1 MiB: 950 + 947 + 189 frames (aggregated: 865 + 857 + 364); default: 1019 + 1019 + 48
    features_ragged_host: ((2086, (32, 6, 6), 0, 1, (3, 3, 0, 3)), (2086, (32, 2, 2), 0, 1, (3, 3, 0, 3))),
    segment_vectors_ragged_host: ((2086, (32, 12, 12), 0, 1, (3, 3, 0, 6)), (2086, (32, 2, 2), 0, 1, (3, 3, 0, 6))),
    # 1 MiB: 921 + 147 frames (aggregated: 871 + 197); default: 1068
    features_ragged_dev: ((1068, (32, 5, 5), 0, 1, (2, 2, 0, 2)), (1068, (32, 34, 34), 0, 1, (1, 1, 0, 1))),
    segment_vectors_ragged_dev: ((1068, (32, 7, 7), 0, 1, (2, 2, 0, 4)), (1068, (32, 34, 34), 0, 1, (1, 1, 0, 2))),
    # no launch of these forms is timed (the device STFT and Welch forms time theirs), so nothing is counted; their outputs must
    # still not depend on the limit
    stft_host_tables: (((0, 0, 0, 0),), ((0, 0, 0, 0),)),
    psd_welch_host_tables: (((0, 0, 0, 0),), ((0, 0, 0, 0),)),
    spectral_contrast_from_mag: (((0, 0, 0, 0),), ((0, 0, 0, 0),)),
}


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


@pytest.mark.parametrize("call", list(PINS), ids=lambda c: c.__name__)
def test_chunk_pins(eng, call):
    lib = eng.lib
    gpu = eng.test_backend == "gpu"
    feature = len(PINS[call][0]) > 1
    outs, pins = [], []
    lib.dll.syg_debug_set_resident_min_groups(MIN_GROUPS)
    try:
        eng.profile_enable(True)
        for limit in (SMALL, DEFAULT):
            eng.set_workspace_limit(limit)
            eng.profile_read(reset=True)
            outs.append(call(eng))
            launches = tuple(n for _, n in eng.profile_read(reset=True).values())
            getters = (lib.last_feature_frames(), lib.last_finalize(), int(lib.dll.syg_debug_last_features_resident()),
                       int(lib.dll.syg_debug_last_mel_form())) if feature else ()
            pins.append(getters + (launches,))
    finally:
        eng.profile_enable(False)
        eng.profile_read(reset=True)
        eng.set_workspace_limit(DEFAULT)
        lib.dll.syg_debug_set_resident_min_groups(-1)
    # the emulator's events are null: nothing is timed or counted there
    expected = [pin if gpu else pin[:-1] + ((0, 0, 0, 0),) for pin in PINS[call]]
    assert pins == expected
    assert np.array_equal(outs[0], outs[1], equal_nan=True)
