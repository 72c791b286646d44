"""The mixed-radix kernels (syg_mixed.cuh) at the FP32 noise floor across every radix, pass position, CTA width and size limit.

Every transform length outside the power-of-two kernels (13-smooth, 8 up to the shared-memory limit) runs on ``frame_mixed_kernel``
(features, STFT) or ``welch_mixed_kernel``.  Which passes a length gets is decided on the host (``mixed_plan_of`` in syg_api.cu,
``sygplan::factorize_smooth``, ``sygdev::mixed_layout``, ``mixed_threads`` in syg_launch_mixed.cu); this file restates that planner
in Python, checks the restatement against the library for every length up to 30 000, and uses it to choose a cover set of lengths
that reaches every radix before and after a twiddled pass, the squares and cubes of the generic O(R^2) radices, each CTA width on
both sides of its boundaries in both parities, odd transforms packed inside even ones, the tiny lengths and the largest length of
each entry point.  On the cover set the STFT (all three output kinds), Welch and the feature rows are held to the yardstick of
test_noise_floor (DESIGN.md 2): ``max_k |X^ - X64| <= 8 floor`` per frame.  On the B200 every served STFT length and every odd
Welch length is swept.
"""
import collections

import numpy as np
import pytest

from backends import BACKENDS, get_engine
from oracle import sygnals_oracle as orc
from sygnals_b200 import _ffi
from sygnals_b200.utils import synth
from test_noise_floor import (ALL16, C, EPS32, K_SPREAD, SIGNALS, TIME_ROWS, Yardstick, _mels, check_dominant, check_floor, check_sideband,
                              envelope_rows, make_signal, make_units, tone_bins, welch_yardstick, yardstick_rows)
from test_parity_cabi import check_rows, oracle_rows, row_tol


@pytest.fixture(params=BACKENDS)
def eng(request):
    return get_engine(request.param)


MAG, PW, CX = _ffi.OUT_MAGNITUDE, _ffi.OUT_POWER, _ffi.OUT_COMPLEX
KINDS = (CX, MAG, PW)
KIND_NAME = {CX: "complex", MAG: "magnitude", PW: "power"}
STFT_MIXED = 5                                      # syg_debug_last_stft_path of frame_mixed_kernel<MODE_STFT>


# ------------------------------------------------------------------------------------------------ the floor rules of test_noise_floor
def check_welch_floor(psd, y, fs, nperseg, noverlap, nfft, detrend, scaling, signal):
    """test_welch_floor's bound for psd [units, B] of the units y [units, L], in either scaling (0 density, 1 spectrum): with
    |X^_s - X64_s| <= C floor_s per segment, the averaged one-sided PSD is off by at most scale * mean_s(2 |X64_s| C floor_s +
    (C floor_s)^2) plus the float32 rounding of the power and the average; the -90 dB sideband of units 0 and 2 within 1 %.
    Returns the ratios per unit."""
    ratios = []
    for u in range(len(y)):
        _, ref = orc.compute_psd_welch(y[u].astype(np.float64), fs=fs, nperseg=nperseg, noverlap=noverlap, nfft=nfft,
                                       detrend="constant" if detrend else False, scaling=("density", "spectrum")[scaling])
        X64, floor, scale = welch_yardstick(y[u], fs, nperseg, noverlap, nfft, detrend, scaling)
        P64 = (scale[:, None] * np.abs(X64) ** 2).mean(axis=1)
        np.testing.assert_allclose(P64, ref, rtol=1e-9, atol=1e-12 * ref.max())        # the float64 leg is scipy's Welch
        if not (floor > 0).any():
            assert (psd[u] == 0).all(), f"unit {u}: all-zero segments give a non-zero PSD"
            continue
        unit = scale * (2 * np.abs(X64) * floor + floor ** 2).mean(axis=1)   # the bound per unit of C
        err = np.maximum(np.abs(psd[u] - ref) - 4 * EPS32 * ref, 0.0)
        ratio = (err / np.maximum(unit, 1e-300)).max()
        ratios.append(float(ratio))
        bound = scale * (2 * np.abs(X64) * C * floor + (C * floor) ** 2).mean(axis=1) + 4 * EPS32 * ref
        bad = np.abs(psd[u] - ref) > bound
        assert not bad.any(), f"nfft {nfft} unit {u}: {bad.sum()} PSD bins beyond {C} x the FP32 floor ({ratio:.2f} x)"
        if signal == "sideband" and u != 1:
            _, ks = tone_bins(nfft)
            off = abs(np.sqrt(psd[u][ks] / ref[ks]) - 1.0)
            assert off <= 1e-2, f"unit {u}: -90 dB sideband off by {100 * off:.3f} %"
    return ratios


def check_features_floor(out, y, sr, feats, n_fft, hop, fp):
    """test_features_floor's rule for out [units, rows, T] of the units y [units, L]: time rows at the parity bars; spectral rows
    at the parity bar plus max(4 x the yardsticks' spread, their spread at C x their error), contrast also within the envelope of
    the transform bound; the dominant frequency tie-aware; all-zero units at their exact values."""
    bin_hz, nyq = sr / n_fft, sr / 2
    for u in range(len(y)):
        names, ref, spread = yardstick_rows(y[u], sr, feats, n_fft, hop, fp)
        _, _, spread_c = yardstick_rows(y[u], sr, feats, n_fft, hop, fp, gain=C)
        if "spectral_contrast" in feats:
            _, env = envelope_rows(y[u], sr, feats, n_fft, hop, fp)
            con = [i for i, n in enumerate(names) if n.startswith("contrast_")]
            spread_c[con] = np.maximum(spread_c[con], env[con])
        got = out[u].astype(np.float64)
        assert got.shape == ref.shape
        ys = Yardstick(y[u], n_fft, hop)
        ti = [i for i, n in enumerate(names) if n in TIME_ROWS]
        check_rows([names[i] for i in ti], got[ti], ref[ti], bin_hz=bin_hz, nyq=nyq)
        for i, n in enumerate(names):
            if n in TIME_ROWS:
                continue
            what = f"n_fft {n_fft} unit {u} {n}"
            if n == "dominant_frequency":
                check_dominant(got[i], ys, bin_hz, what)
                continue
            d = np.abs(got[i] - ref[i])
            tol = row_tol(n, ref[i], bin_hz=bin_hz, nyq=nyq) + np.maximum(K_SPREAD * spread[i], spread_c[i])
            assert np.isfinite(got[i]).all(), f"{what}: not finite"
            bad = d > tol
            assert not bad.any(), f"{what}: frame {np.argmax(d - tol)} off by {d[bad][0]:.4g} (float64 {ref[i][bad][0]:.6g})"
        if not y[u].any():                             # exact expectations of all-zero frames (frequency_domain.py, time_domain.py)
            d = dict(zip(names, got))
            for n, v in (("spectral_centroid", 0.0), ("spectral_bandwidth", 0.0), ("spectral_flatness", 0.0), ("dominant_frequency", 0.0),
                         ("rms_energy", 0.0), ("crest_factor", 0.0), ("spectral_rolloff", sr * (n_fft // 2) / n_fft)):
                if n in d:
                    assert (d[n] == np.float32(v)).all(), f"{n} of silence: {np.unique(d[n])}"


# ------------------------------------------------------------------------------------------------ 1. the planner, restated
SMEM_LIMIT = 227 * 1024                             # kMaxDynSmem (syg_api.cu)
PLAN_THREADS = 256                                  # mixed_plan_of sizes the layout at kThreads
Plan = collections.namedtuple("Plan", "n L packed radices nt")


def factorize_smooth(L):
    """sygplan::factorize_smooth: fours first, then 2, 3, 5, 7, 11, 13; None when L has a larger prime factor."""
    if L < 1:
        return None
    r = []
    while L % 4 == 0:
        r.append(4)
        L //= 4
    for p in (2, 3, 5, 7, 11, 13):
        while L % p == 0:
            r.append(p)
            L //= p
    return tuple(r) if L == 1 else None


def mixed_layout_bytes(L, B, features, nt=PLAN_THREADS):
    """sygdev::mixed_layout(...).bytes: two float2 buffers of L, then (features only) the padded power row, contrast candidates and
    unit maxima, then the reduction scratch: nt/32 doubles, plus nt doubles of scan results for the feature epilogue."""
    off_cand = 4 * L + ((B + (B >> 5) + 1) if features else 0)
    off_smax = off_cand + ((nt // 32) * 32 if features else 0)
    off_dsc = (off_smax + 4 + 1) // 2 * 2
    return 4 * (off_dsc + 2 * (nt // 32 + (nt if features else 0)))


def mixed_threads(L):
    """syglaunch::mixed_threads"""
    return 64 if L <= 256 else 128 if L <= 1024 else 256


def assert_width(eng, n, features=False):
    """the launch ran at the CTA width the mirror gives n"""
    got, want = eng.lib.dll.syg_debug_last_mixed_threads(), mixed_plan(n, features).nt
    assert got == want, f"length {n} ran {got} threads per CTA, the planner says {want}"


def native_pow2(n):
    return 32 <= n <= 8192 and n & (n - 1) == 0


def mixed_plan(n, features):
    """mixed_plan_of: a Plan, or the phrase of the library's refusal"""
    if n < 8:
        return "below 8"
    packed = n % 2 == 0
    L = n // 2 if packed else n
    r = factorize_smooth(L)
    if r is None or len(r) > 24:
        return "prime factors"
    if mixed_layout_bytes(L, n // 2 + 1, features) > SMEM_LIMIT:
        return "does not fit in shared memory"
    return Plan(n, L, packed, r, mixed_threads(L))


def served_mixed(features, lo=8, hi=30000):
    """every length the mixed-radix kernels serve (the power-of-two kernels keep 32 ... 8192)"""
    return [n for n in range(lo, hi + 1) if not native_pow2(n) and isinstance(mixed_plan(n, features), Plan)]


def limits(features, parity):
    """(largest served, smallest refused) smooth length of the parity"""
    ns = [n for n in range(8 + parity, 30001, 2) if factorize_smooth(n // 2 if n % 2 == 0 else n)]
    ok = [n for n in ns if isinstance(mixed_plan(n, features), Plan)]
    return max(ok), min(n for n in ns if n > max(ok))


# entry point -> (largest served, smallest refused) per parity; DESIGN 4.4b states the same numbers
BOUNDARY = {("stft", "even"): (29040, 29106), ("stft", "odd"): (14175, 14553),
            ("features", "even"): (22750, 22880), ("features", "odd"): (12675, 12705)}


def test_boundary_table_is_the_planners():
    for (ep, par), want in BOUNDARY.items():
        assert limits(ep == "features", par == "odd") == want, (ep, par)
    assert mixed_layout_bytes(14400, 14401, False) <= SMEM_LIMIT     # 28 800, the length DESIGN has always promised


def _plan_call(eng, entry, n):
    """a request of no units: the library plans the transform (host code) and launches nothing"""
    y = np.zeros(1, np.float32)
    if entry == "stft":
        eng.stft_host(y, eng.units_clips(0, n), n, n, n, 0, True, 0, PW)
    elif entry == "welch":
        eng.psd_welch_host(y, eng.units_clips(0, n), 1.0, 0, n, 0, n, True, 0)
    else:
        eng.features_host(y, eng.units_clips(0, n), _ffi.make_params(eng.lib, 22050, ["rms_energy"], n, n))


@pytest.mark.parametrize("entry", ["stft", "welch", "features"])
def test_planner_mirror_matches_library(entry):
    """For every n in 1 ... 30 000: the library serves n exactly where the mirror does, and refuses the rest with the mirror's
    reason.  A private context keeps the window and twiddle tables of the ~1 000 served lengths out of the shared engine."""
    base = get_engine("emu")
    eng = _ffi.Engine(0, base.lib)
    try:
        # a zero-unit request stops after planning: it launches nothing, so it cannot differ from a request that runs
        out = eng.stft_host(np.zeros(1, np.float32), eng.units_clips(0, 1000), 1000, 250, 1000)
        assert out.shape == (0, 501, 5)
        mismatch = []
        for n in range(1, 30001):
            p = "native" if native_pow2(n) else mixed_plan(n, entry == "features")
            try:
                _plan_call(eng, entry, n)
                got = None
            except NotImplementedError as e:
                got = str(e)
            if isinstance(p, str) and p != "native":
                if got is None or p not in got:
                    mismatch.append((n, p, got))
            elif got is not None:
                mismatch.append((n, "served", got))
        assert not mismatch, f"{len(mismatch)} lengths differ, first {mismatch[:5]}"
    finally:
        eng.close()


@pytest.mark.parametrize("entry", ["stft", "welch", "features"])
def test_size_limits(eng, entry):
    """The largest served and the smallest refused length of each parity, with the refusal message."""
    key = "features" if entry == "features" else "stft"
    for par in ("even", "odd"):
        top, refused = BOUNDARY[key, par]
        _plan_call(eng, entry, top)
        with pytest.raises(NotImplementedError, match=f"={refused}: the transform does not fit in shared memory"):
            _plan_call(eng, entry, refused)
    with pytest.raises(NotImplementedError, match="below 8"):
        _plan_call(eng, entry, 7)
    with pytest.raises(NotImplementedError, match="prime factors"):
        _plan_call(eng, entry, 2 * 17)


# ------------------------------------------------------------------------------------------------ 2. the cover set
TINY = (8, 9, 10, 12, 15, 16, 22, 26)
WIDTH_EDGES = (256, 1024)                           # mixed_threads' boundaries in L


def parity(p):
    return "even" if p.packed else "odd"


def rows_of(p):
    """the coverage rows plan p witnesses"""
    rows = set()
    Ns = 1
    for R in p.radices:
        rows.add(f"radix {R} Ns=1" if Ns == 1 else f"radix {R} Ns>1")
        Ns *= R
    cnt = collections.Counter(p.radices)
    rows |= {f"{R}^2" for R in (3, 5, 7, 11, 13) if cnt[R] >= 2}
    rows |= {f"{R}^3" for R in (11, 13) if cnt[R] >= 3}
    rows.add(f"{p.nt} threads {parity(p)}")
    for b in WIDTH_EDGES:
        if b - b // 4 < p.L <= b:
            rows.add(f"L in ({b - b // 4}, {b}] {parity(p)}")
        if b < p.L <= b + b // 4:
            rows.add(f"L in ({b}, {b + b // 4}] {parity(p)}")
    if p.packed and p.L % 2:
        rows.add("odd L packed")
    if p.n in TINY:
        rows.add(f"n={p.n}")
    rows |= {f"largest {ep} {par}" for (ep, par), (top, _) in BOUNDARY.items() if p.n == top}
    return rows


REQUIRED = ({f"radix {R} Ns{s}" for R in (2, 3, 4, 5, 7, 11, 13) for s in ("=1", ">1")}
            | {f"{R}^2" for R in (3, 5, 7, 11, 13)} | {"11^3", "13^3"}
            | {f"{nt} threads {par}" for nt in (64, 128, 256) for par in ("even", "odd")}
            | {f"L in ({lo}, {hi}] {par}" for b in WIDTH_EDGES for lo, hi in ((b - b // 4, b), (b, b + b // 4)) for par in ("even", "odd")}
            | {"odd L packed"} | {f"n={n}" for n in TINY}
            | {f"largest {ep} {par}" for ep, par in BOUNDARY})

# 231 = 3 7 11 and 273 = 3 7 13 put odd lengths on both sides of L = 256; 1001 / 1029 / 1155 around 1024; 504 / 520 and 2000 / 2080
# the even ones.  The largest lengths come from the mirror.
SEED = (8, 9, 10, 12, 15, 16, 22, 26, 121, 143, 169, 231, 242, 273, 286, 338, 504, 520, 1001, 1029, 1155, 1331, 2000, 2080, 2197, 2662,
        3003, 4394, 9009, 12288, 28800)
COVER = sorted(set(SEED) | {limits(False, 0)[0], limits(False, 1)[0], limits(True, 0)[0], limits(True, 1)[0]})
FEATURE_MAX = {limits(True, 0)[0], limits(True, 1)[0]}


def plan_for(n):
    """the STFT / Welch plan of n, or the feature plan of the features maxima"""
    return mixed_plan(n, n in FEATURE_MAX)


def test_cover_set_witnesses_every_row():
    plans = [plan_for(n) for n in COVER]
    assert all(isinstance(p, Plan) for p in plans), [p for p in plans if not isinstance(p, Plan)]
    witnessed = set().union(*map(rows_of, plans))
    missing = REQUIRED - witnessed
    assert not missing, f"no cover length witnesses {sorted(missing)}"
    for n in COVER:                                       # and every cover length is there for a reason
        assert rows_of(plan_for(n)) & REQUIRED, n


# ------------------------------------------------------------------------------------------------ 3. STFT floor
def noise_units(n_units, L, seed):
    """seeded N(0, 1) unit, the same at 1e-3, and a silent unit"""
    s = np.random.default_rng(seed).standard_normal(L).astype(np.float32)
    return np.ascontiguousarray(np.stack([s, s * np.float32(1e-3), np.zeros(L, np.float32)])[:n_units])


def stft_floor(eng, y, n, hop, kinds, signal, win_length=None, center=True, pad_mode="constant"):
    """STFT of the units y [U, L] for each output kind on the mixed-radix kernel, against the yardstick; returns the largest ratio"""
    ratios = []
    U, L = y.shape
    for kind in kinds:
        out = eng.stft_host(y.ravel(), eng.units_clips(U, L), n, hop, win_length or n, 0, center, _ffi.PAD_IDS[pad_mode], kind)
        assert eng.lib.dll.syg_debug_last_stft_path() == STFT_MIXED, f"ran stft path {eng.lib.dll.syg_debug_last_stft_path()}"
        assert_width(eng, n)
        for u in range(U):
            ys = Yardstick(y[u], n, hop, win_length, center, pad_mode)
            assert out[u].shape == ys.X64.shape
            what = f"n_fft {n} {KIND_NAME[kind]} unit {u}"
            check_floor(out[u], ys, kind, ratios, what)
            if signal == "sideband" and u != 1:
                check_sideband(out[u], ys, kind, n, what)
    return max(ratios)


@pytest.mark.parametrize("n", COVER)
def test_stft_floor_random(eng, n, record_property):
    """a seeded random unit, the same at 1e-3 and a silent one, about three frames each, all three output kinds"""
    L, hop = n + n // 2, n // 2 + 1
    record_property("floor_ratio", stft_floor(eng, noise_units(3, L, n), n, hop, KINDS, "random"))


@pytest.mark.parametrize("n", COVER)
def test_stft_floor_signals(eng, n, record_property):
    """the tonal, DC, impulse, square, near-silent and -90 dB sideband signals of test_noise_floor: two or three interior frames"""
    L, hop = 2 * n + 4, max(1, n // 2 - 1)
    ratio = 0.0
    for i, signal in enumerate(SIGNALS):
        y = make_units(signal, L, 22050, n)
        kinds = KINDS if signal == "sideband" else (KINDS[i % 3],)
        ratio = max(ratio, stft_floor(eng, y, n, hop, kinds, signal))
    record_property("floor_ratio", ratio)


# (n_fft, hop, win_length, center, pad_mode): odd lengths framed every way the STFT allows; 441 / 400 centres the window at lpad 20
FRAMING = [(441, 110, 400, True, "constant"), (441, 147, None, False, "constant"), (1155, 300, None, True, "reflect"),
           (273, 91, 200, True, "reflect"), (2197, 700, 2000, False, "constant"), (286, 71, 255, True, "constant"),
           (14175, 5000, 14000, True, "reflect")]


@pytest.mark.parametrize("n,hop,wl,center,pad", FRAMING, ids=[f"{f[0]}_{f[2]}_{'c' if f[3] else 'nc'}_{f[4]}" for f in FRAMING])
def test_stft_floor_framing(eng, n, hop, wl, center, pad, record_property):
    L = 2 * n + 3
    y = noise_units(2, L, n + 1)
    y[1] = make_signal("sideband", L, 22050, n)
    record_property("floor_ratio", stft_floor(eng, y, n, hop, KINDS, "random", wl, center, pad))


# ------------------------------------------------------------------------------------------------ 4. Welch floor
# (name, nperseg, nfft): odd and even nfft at each CTA width, then nperseg < nfft for every parity mix
WELCH = [("w64_even", 504, 504), ("w64_odd", 231, 231), ("w128_even", 520, 520), ("w128_odd", 1001, 1001),
         ("w256_even", 2080, 2080), ("w256_odd", 1155, 1155), ("odd_in_even", 143, 286), ("even_in_odd", 1000, 1155),
         ("odd_in_odd", 945, 1001), ("even_in_even", 400, 520), ("tiny_odd", 9, 15), ("tiny_even", 8, 10)]


def welch_units(signal, L, fs, nfft):
    if signal == "random":
        return noise_units(3, L, nfft)
    return make_units(signal, L, fs, nfft)


def check_nyquist(psd, y, fs, nperseg, noverlap, nfft, detrend, scaling):
    """The one-sided doubling: DC single, Nyquist single for even nfft, the last bin doubled for odd nfft.  A wrong factor is off
    by 2; the floor bound has already held the bins to their precision."""
    for u in range(len(y)):
        X64, _, scale = welch_yardstick(y[u], fs, nperseg, noverlap, nfft, detrend, scaling)
        P64 = (scale[:, None] * np.abs(X64) ** 2).mean(axis=1)
        for k in (0, len(P64) - 1):
            if P64[k] > 1e-6 * P64.max():
                r = psd[u][k] / P64[k]
                assert abs(r - 1.0) < 0.25, f"unit {u} bin {k} of nfft {nfft}: {r:.3f} x the one-sided value"


@pytest.mark.parametrize("scaling", [0, 1], ids=["density", "spectrum"])
@pytest.mark.parametrize("detrend", [True, False], ids=["detrend", "raw"])
@pytest.mark.parametrize("signal", ["random", "dc_noise", "sideband"])
@pytest.mark.parametrize("arm", WELCH, ids=[a[0] for a in WELCH])
def test_welch_floor_mixed(eng, arm, signal, detrend, scaling, record_property):
    name, nperseg, nfft = arm
    fs = 25600
    noverlap = nperseg // 2
    L = 3 * nperseg + 5
    y = welch_units(signal, L, fs, nfft)
    psd, st = eng.psd_welch_host(y.ravel(), eng.units_clips(3, L), fs, 0, nperseg, noverlap, nfft, detrend, scaling, stats=True)
    assert eng.lib.dll.syg_debug_last_welch_path() == _ffi.WELCH_MIXED
    assert_width(eng, nfft)
    ratios = check_welch_floor(psd, y, fs, nperseg, noverlap, nfft, detrend, scaling, signal)
    check_nyquist(psd, y, fs, nperseg, noverlap, nfft, detrend, scaling)
    for u in range(3):                                                # rms, crest, peak of the whole unit
        x = y[u].astype(np.float64)
        rms = np.sqrt(np.mean(x ** 2))
        np.testing.assert_allclose(st[u], [rms, orc.crest_factor(x), orc.peak_amplitude(x)], rtol=1e-6, atol=0)
    record_property("floor_ratio", max(ratios, default=0.0))


@pytest.mark.parametrize("signal", ["random", "dc_noise", "sideband"])
@pytest.mark.parametrize("par", ["even", "odd"])
def test_periodogram_largest(eng, par, signal, record_property):
    """one segment of the largest served length of each parity (compute_psd_periodogram)"""
    nfft = BOUNDARY["stft", par][0]
    fs = 25600
    y = welch_units(signal, nfft, fs, nfft)
    psd = eng.psd_welch_host(y.ravel(), eng.units_clips(3, nfft), fs, 0, nfft, 0, nfft, True, 0)
    assert eng.lib.dll.syg_debug_last_welch_path() == _ffi.WELCH_MIXED
    assert_width(eng, nfft)
    for u in range(3):
        _, ref = orc.compute_psd_periodogram(y[u].astype(np.float64), fs=fs)
        np.testing.assert_allclose(ref, orc.compute_psd_welch(y[u].astype(np.float64), fs=fs, nperseg=nfft, noverlap=0)[1], rtol=1e-12,
                                   atol=1e-300)
    ratios = check_welch_floor(psd, y, fs, nfft, 0, nfft, True, 0, signal)
    check_nyquist(psd, y, fs, nfft, 0, nfft, True, 0)
    record_property("floor_ratio", max(ratios, default=0.0))


# ------------------------------------------------------------------------------------------------ 5. features
# one length per CTA width x parity (1001 = 7 11 13 also runs radix 11 and 13 after twiddled passes), and the features maxima
FEATURE_LENGTHS = [286, 231, 520, 1001, 2080, 1155, *sorted(FEATURE_MAX)]


def test_feature_lengths_cover_widths():
    plans = [mixed_plan(n, True) for n in FEATURE_LENGTHS]
    assert {(p.nt, parity(p)) for p in plans} == {(nt, par) for nt in (64, 128, 256) for par in ("even", "odd")}
    assert {"radix 11 Ns>1", "radix 13 Ns>1"} <= set().union(*map(rows_of, plans))
    assert {"largest features even", "largest features odd"} <= set().union(*map(rows_of, plans))


@pytest.mark.parametrize("n", FEATURE_LENGTHS)
def test_features_floor_mixed(eng, n):
    """All 16 kernelled features on three units (a mixture, silence, a -90 dB sideband) at the floor rule of test_features_floor;
    the ragged launch of the same units gives the same bits."""
    sr = 22050
    hop = n // 3 + 1
    L = 2 * n + hop + 3
    y = np.stack([synth.mixture(L, sr, seed=n), np.zeros(L, np.float32), make_signal("sideband", L, sr, n)]).astype(np.float32)
    fp = _mels(n)
    p = _ffi.make_params(eng.lib, sr, ALL16, n, hop, feature_params=fp)
    out = eng.features_host(y.ravel(), eng.units_clips(3, L), p)
    assert eng.lib.dll.syg_debug_last_feature_kernel() == _ffi.FK_MIXED
    assert_width(eng, n, features=True)
    check_features_floor(out, y, sr, ALL16, n, hop, fp)
    rag = eng.features_ragged_host(y.ravel(), eng.ragged_units([0, L, 2 * L], [L, L, L], 3 * L), p)
    assert eng.lib.dll.syg_debug_last_feature_kernel() == _ffi.FK_MIXED
    uni = out.transpose(1, 0, 2).reshape(out.shape[1], -1)
    assert rag.shape == uni.shape
    assert np.array_equal(rag.view(np.uint32), uni.view(np.uint32)), "ragged launch differs from the uniform launch"


# ------------------------------------------------------------------------------------------------ 6. every served length (B200)
def sweep_stft(eng, lengths):
    """power STFT of one seeded random unit of about three frames per length; the largest ratio per (radix, CTA width)"""
    worst = collections.defaultdict(float)
    bad = []
    for n in lengths:
        p = mixed_plan(n, False)
        L, hop = n + n // 2, n // 2 + 1
        y = noise_units(1, L, n)
        out = eng.stft_host(y.ravel(), eng.units_clips(1, L), n, hop, n, 0, True, 0, PW)
        assert eng.lib.dll.syg_debug_last_stft_path() == STFT_MIXED, n
        assert_width(eng, n)
        rec = []
        try:
            check_floor(out[0], Yardstick(y[0], n, hop), PW, rec, f"n_fft {n}")
        except AssertionError as e:
            bad.append(str(e))
        for R in set(p.radices):
            worst[R, p.nt] = max(worst[R, p.nt], max(rec, default=float("inf")))
    return worst, bad


def sweep_welch(eng, lengths):
    worst = collections.defaultdict(float)
    bad = []
    fs = 25600
    for n in lengths:
        p = mixed_plan(n, False)
        L = 2 * n
        y = noise_units(1, L, n)
        psd = eng.psd_welch_host(y.ravel(), eng.units_clips(1, L), fs, 0, n, n // 2, n, True, 0)
        assert eng.lib.dll.syg_debug_last_welch_path() == _ffi.WELCH_MIXED, n
        assert_width(eng, n)
        try:
            r = check_welch_floor(psd, y, fs, n, n // 2, n, True, 0, "random")
        except AssertionError as e:
            bad.append(f"nfft {n}: {e}")
            r = [float("inf")]
        for R in set(p.radices):
            worst[R, p.nt] = max(worst[R, p.nt], max(r))
    return worst, bad


def record_worst(record_property, what, worst):
    for (R, nt), v in sorted(worst.items()):
        record_property(f"{what}_radix{R}_nt{nt}", round(v, 3))


@pytest.mark.gpu
def test_every_served_stft_length(record_property):
    lengths = served_mixed(False)
    assert len(lengths) == 1064
    worst, bad = sweep_stft(get_engine("gpu"), lengths)
    record_worst(record_property, "stft", worst)
    assert not bad, f"{len(bad)} lengths beyond {C} x the floor: {bad[:5]}"


@pytest.mark.gpu
def test_every_odd_welch_length(record_property):
    lengths = [n for n in served_mixed(False) if n % 2]
    assert len(lengths) == 218
    worst, bad = sweep_welch(get_engine("gpu"), lengths)
    record_worst(record_property, "welch", worst)
    assert not bad, f"{len(bad)} lengths beyond {C} x the floor: {bad[:5]}"


# ------------------------------------------------------------------------------------------------ regressions
def test_entropy_bin_edges_round_like_linspace(eng):
    """frame_length 2080, frames 1 and 6 of the -90 dB sideband signal: the zeros of the padding lie on a histogram edge.  numpy's
    linspace rounds idx * step before adding the first edge; with the two fused into one multiply-add the B200 put those zeros in
    the next bin and the entropy off by 1.4e-3."""
    sr, n = 22050, 2080
    hop = n // 3 + 1
    L = 2 * n + hop + 3
    y = make_signal("sideband", L, sr, n)
    p = _ffi.make_params(eng.lib, sr, ["signal_entropy"], n, hop)
    out = eng.features_host(y, eng.units_clips(1, L), p)
    names, ref = oracle_rows(y, sr, ["signal_entropy"], n, hop)
    assert names == ["signal_entropy"]
    np.testing.assert_allclose(out[0], ref, rtol=0, atol=1e-6)

