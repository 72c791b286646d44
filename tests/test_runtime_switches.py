"""Every arm of the run-time comparison switches (the SYGB200_* variables the library reads once per process, DESIGN.md 6) against
the default arm and the float64 oracle.

A switch is cached in a function-local static on first use, so one process sees one arm.  Each arm therefore runs in a child
process: this module is also the worker (``python test_runtime_switches.py <backend> <out.npz> <case,...>``).  The child's
environment is the parent's without any SYGB200_* variable (SYGB200_DEVICE excepted), plus the one switch under test; the default
arm runs the same way, so a switch exported in the caller's shell cannot turn the baseline into the arm under test.  A child
writes each output and the debug getters read right after the call that produced it to an .npz; the parent compares.

Each case asserts three things:
* the switched arm ran: the getter of the switched child shows the arm, and the default child's shows the default kernel;
* the switched output matches the oracle at the tolerances of test_parity_cabi.py;
* the switched output equals the default output bit for bit where both arms do the same arithmetic, else within the bar given in
  the switch's table entry (with the reason).
"""
import os
import re
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for _p in (ROOT, HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from backends import BACKENDS  # noqa: E402
from sygnals_b200 import _ffi  # noqa: E402

CFG4 = ["mfcc", "spectral_contrast", "spectral_centroid", "spectral_rolloff", "rms_energy", "crest_factor"]
CFG4_REORDERED = ["rms_energy", "mfcc", "crest_factor", "spectral_contrast", "spectral_rolloff", "spectral_centroid"]
NO_RESIDENT = 1 << 30           # syg_debug_set_resident_min_groups: the two-kernel path whatever the batch


# ------------------------------------------------------------------------------------------------ cases
# features: (sr, n_fft, hop, features, feature_params, form, units, resident min groups or None)
#   form "uniform": units = (n clips, clip length); "ragged": units = clip lengths; "vectors": uniform units -> segment vectors (mean)
#   units None: enough units for FIN_CTAS=1 to give each CTA at least 5 tiles in the last chunk of the host pipeline, which holds
#   half the units (the count depends on the device's SMs): units of 16000 samples, or for "ragged" clips of 16000 / 7000 / 300 /
#   11000 samples in turn
def _f(sr, fl, hop, feats, fp, form="uniform", units=(2, 9000), res=NO_RESIDENT):
    return dict(kind="features", sr=sr, fl=fl, hop=hop, feats=feats, fp=fp, form=form, units=units, res=res)


M128_20 = {"mfcc": {"n_mels": 128, "n_mfcc": 20}}
FEATURE_CASES = {
    "mfcc512": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, units=(5, 4000)),
    "mfcc512_resident": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, units=(7, 4000), res=1),
    "mfcc1024": _f(22050, 1024, 256, ["mfcc", "rms_energy"], {"mfcc": {"n_mels": 64}}, units=(2, 5000)),
    "cfg4": _f(44100, 2048, 512, CFG4, None),
    "cfg4_reordered": _f(44100, 2048, 512, CFG4_REORDERED, None),
    "cfg4_at_22k": _f(22050, 2048, 512, CFG4, None),
    "cfg1": _f(22050, 2048, 512, ["mfcc", "rms_energy"], M128_20),
    "cfg1_at_48k": _f(48000, 2048, 512, ["mfcc", "rms_energy"], M128_20),
    "cfg4_ragged": _f(44100, 2048, 512, CFG4, None, form="ragged", units=(9000, 3000, 700, 12000)),
    "cfg4_vectors": _f(44100, 2048, 512, CFG4, None, form="vectors"),
    "cfg1_ragged": _f(22050, 2048, 512, ["mfcc", "rms_energy"], M128_20, form="ragged", units=(5000, 9000, 300)),
    # cfg3's shape on the resident kernel: 11 units (no group size divides it), unit 2 silent
    "cfg3_resident": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, units=(11, 16000), res=1),
    # finalize tile heights: 64 by default for <= 64 mels with MFCCs, else 32
    "fin_mel40": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, units=(5, 4000)),
    "fin_mel128": _f(22050, 1024, 256, ["mfcc"], {"mfcc": {"n_mels": 128}}, units=(3, 5000)),
    "fin_contrast": _f(22050, 1024, 256, ["spectral_contrast"], None, units=(3, 5000)),
    "fin_mfcc_contrast": _f(16000, 512, 160, ["mfcc", "spectral_contrast"], {"mfcc": {"n_mels": 40}}, units=(4, 4000)),
    "fin_mel40_vectors": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, form="vectors", units=(5, 4000)),
    "fin_mel128_vectors": _f(22050, 1024, 256, ["mfcc"], {"mfcc": {"n_mels": 128}}, form="vectors", units=(3, 5000)),
    "fin_mel40_ragged": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, form="ragged", units=(4000, 100, 2500, 7000)),
    "fin_mel128_ragged": _f(22050, 1024, 256, ["mfcc"], {"mfcc": {"n_mels": 128}}, form="ragged", units=(5000, 1200, 3000)),
    "fin_mfcc_contrast_ragged": _f(16000, 512, 160, ["mfcc", "spectral_contrast"], {"mfcc": {"n_mels": 40}}, form="ragged",
                                   units=(4000, 900, 6000)),
    # many tiles per CTA: cfg3-shaped units (T = 101, tiles of 64) and a 128-mel plan (tiles of 32)
    "fin_many_tiles": _f(16000, 512, 160, ["mfcc"], {"mfcc": {"n_mels": 40}}, units=None),
    "fin_many_tiles_mel128": _f(16000, 1024, 256, ["mfcc"], {"mfcc": {"n_mels": 128}}, units=None),
    "fin_many_tiles_ragged": _f(16000, 1024, 256, ["mfcc", "spectral_contrast"], {"mfcc": {"n_mels": 128}}, form="ragged", units=None),
}


def _s(n_fft, hop, L, n, kinds=("complex", "magnitude", "power"), pad=0):
    return dict(kind="stft", n_fft=n_fft, hop=hop, L=L, n=n, kinds=kinds, pad=pad)


STFT_CASES = {
    # every size of the CTA-cooperative kernel; frame counts that leave partial rounds; reflect padding at three sizes
    "stft32": _s(32, 8, 301, 3), "stft64": _s(64, 16, 777, 2, pad=1), "stft128": _s(128, 32, 1001, 3),
    "stft256": _s(256, 64, 3000, 2), "stft512": _s(512, 128, 4100, 3, pad=1), "stft1024": _s(1024, 256, 5000, 2),
    "stft2048": _s(2048, 512, 9001, 2), "stft4096": _s(4096, 1024, 16000, 2), "stft8192": _s(8192, 2048, 30000, 1, pad=1),
    # warp kernel, real output at n_fft <= 512: frame counts not multiples of 8; odd hops at 256 / 512 keep the ring kernel out
    "real32": _s(32, 8, 300, 5, ("magnitude", "power")), "real64": _s(64, 16, 1000, 7, ("magnitude", "power")),
    "real128": _s(128, 32, 777, 3, ("magnitude", "power")), "real256": _s(256, 63, 1601, 9, ("magnitude", "power")),
    "real512": _s(512, 127, 3000, 11, ("magnitude", "power")),
    # the ring kernel's sizes on aligned units
    "ring256": _s(256, 64, 4000, 3, ("magnitude", "power")), "ring512": _s(512, 128, 4000, 2, ("magnitude", "power")),
    "ring1024": _s(1024, 256, 8000, 3, ("magnitude", "power")), "ring2048": _s(2048, 512, 16000, 2, ("magnitude", "power")),
}


def _w(nfft, nperseg, noverlap, detrend, scaling):
    return dict(kind="welch", nfft=nfft, nperseg=nperseg, noverlap=noverlap, detrend=detrend, scaling=scaling)


WELCH_CASES = {   # every tile size of the warp kernel, with stats; detrend on / off, density / spectrum, nfft > nperseg
    "welch32": _w(32, 32, 16, True, 0), "welch64": _w(64, 64, 0, False, 1), "welch128": _w(128, 128, 64, True, 1),
    "welch256": _w(256, 200, 100, True, 0), "welch512": _w(512, 400, 100, False, 0), "welch1024": _w(1024, 1024, 512, True, 0),
    "welch2048": _w(2048, 2048, 1024, False, 1),
}
CASES = {**FEATURE_CASES, **STFT_CASES, **WELCH_CASES}

# ------------------------------------------------------------------------------------------------ switch table
# getters recorded after every call, in this order
GETTERS = ("feature_kernel", "mel_form", "resident", "fin_tt", "fin_ctas", "fin_tiles", "stft_path", "welch_path")
FK = _ffi
WIDE, WARP, S44, S22, S44L, RES = FK.FK_WARP_WIDE, FK.FK_WARP, FK.FK_SPEC44K, FK.FK_SPEC22K, FK.FK_SPEC44KL, FK.FK_RESIDENT

# switch -> {value: [(case, {getter: (default arm, switched arm)}), ...]}, and how the switched output relates to the default one:
#   "bit": equal bit for bit; "oracle": no bar beyond the oracle; ("atol", x) / ("rtol", x): numpy.allclose-style bars
SWITCHES = {
    # mel form 1 -> 0: the padded tap sweeps sum in another order than the interval form -> oracle only.  With the interval form
    # spec_matches ignores the mel bank, so cfg1's 22.05 kHz and 48 kHz MFCC requests run Spec44k.  With the sweeps it compares the
    # sweep lengths (the only mel constants of a specialisation; the taps come from the plan's tables): the 22.05 kHz bank has
    # Spec22k's and moves there, the 48 kHz bank has Spec44k's and stays.
    "SYGB200_MEL_IV": {
        "0": ("oracle", [("mfcc512", {"mel_form": (1, 0), "feature_kernel": (WARP, WARP)}),
                         ("mfcc512_resident", {"mel_form": (1, 0), "feature_kernel": (RES, RES)}),
                         ("mfcc1024", {"mel_form": (1, 0), "feature_kernel": (WARP, WARP)}),
                         ("cfg4", {"mel_form": (1, 0), "feature_kernel": (S44L, S44L)}),
                         ("cfg4_reordered", {"mel_form": (1, 0), "feature_kernel": (S44, S44)}),
                         ("cfg4_at_22k", {"mel_form": (1, 0), "feature_kernel": (S22, S22)}),
                         ("cfg1", {"mel_form": (1, 0), "feature_kernel": (S44, S22)}),
                         ("cfg1_at_48k", {"mel_form": (1, 0), "feature_kernel": (S44, S44)}),
                         ("cfg4_ragged", {"mel_form": (1, 0), "feature_kernel": (S44L, S44L)})]),
        # =1 keeps the interval form up to n_fft 1024 (same kernel, same output) and the sweeps at 2048
        "1": ("oracle", [("mfcc1024", {"mel_form": (1, 1)}, "bit"),
                         ("cfg4", {"mel_form": (1, 0), "feature_kernel": (S44L, S44L)}),
                         ("cfg4_reordered", {"mel_form": (1, 0), "feature_kernel": (S44, S44)}),
                         ("cfg4_at_22k", {"mel_form": (1, 0), "feature_kernel": (S22, S22)}),
                         ("cfg1", {"mel_form": (1, 0), "feature_kernel": (S44, S22)}),
                         ("cfg1_at_48k", {"mel_form": (1, 0), "feature_kernel": (S44, S44)})]),
    },
    # the plan specialisations fold the same plan into constants: same instructions on the same values
    "SYGB200_NO_SPEC": {
        "1": ("bit", [("cfg4", {"feature_kernel": (S44L, WIDE)}), ("cfg4_reordered", {"feature_kernel": (S44, WIDE)}),
                      ("cfg4_at_22k", {"feature_kernel": (S22, WIDE)}), ("cfg1", {"feature_kernel": (S44, WIDE)}),
                      ("cfg1_at_48k", {"feature_kernel": (S44, WIDE)}), ("cfg4_ragged", {"feature_kernel": (S44L, WIDE)}),
                      ("cfg1_ragged", {"feature_kernel": (S44, WIDE)}), ("cfg4_vectors", {"feature_kernel": (S44L, WIDE)})]),
    },
    "SYGB200_NO_SPECL": {
        "1": ("bit", [("cfg4", {"feature_kernel": (S44L, S44)}), ("cfg4_ragged", {"feature_kernel": (S44L, S44)}),
                      ("cfg4_vectors", {"feature_kernel": (S44L, S44)})]),
    },
    # resident epilogue vs mel workspace + finalize: same energies and dB; as test_resident_units.py
    "SYGB200_NO_RES": {
        "1": (("atol", 2e-5), [("cfg3_resident", {"resident": (1, 0), "feature_kernel": (RES, WARP)}),
                               ("mfcc512_resident", {"resident": (1, 0), "feature_kernel": (RES, WARP)})]),
    },
    # the finalize tile height changes which CTA finishes a frame, not how
    "SYGB200_FIN_TT": {
        "32": ("bit", [("fin_mel40", {"fin_tt": (64, 32)}), ("fin_mfcc_contrast", {"fin_tt": (64, 32)}),
                       ("fin_mel40_vectors", {"fin_tt": (64, 32)}), ("fin_mel40_ragged", {"fin_tt": (64, 32)}),
                       ("fin_mfcc_contrast_ragged", {"fin_tt": (64, 32)})]),
        "64": ("bit", [("fin_mel128", {"fin_tt": (32, 64)}), ("fin_contrast", {"fin_tt": (32, 64)}),
                       ("fin_mel128_vectors", {"fin_tt": (32, 64)}), ("fin_mel128_ragged", {"fin_tt": (32, 64)}),
                       ("fin_mel40_ragged", {"fin_tt": (64, 64)})]),
    },
    # one CTA per SM: the grid-stride loop of finalize_kernel_t covers several tiles per CTA ("ctas < tiles" is checked below)
    "SYGB200_FIN_CTAS": {
        "1": ("bit", [("fin_many_tiles", {"fin_tt": (64, 64)}), ("fin_many_tiles_mel128", {"fin_tt": (32, 32)}),
                      ("fin_many_tiles_ragged", {"fin_tt": (32, 32)})]),
    },
    # CTA-cooperative Welch kernel: another reduction order -> oracle
    "SYGB200_WELCH_BLOCK": {
        "1": ("oracle", [(c, {"welch_path": (FK.WELCH_WARP, FK.WELCH_BLOCK)}) for c in WELCH_CASES]),
    },
    # frame_kernel<MODE_STFT> for every size: its own FFT passes -> oracle
    "SYGB200_STFT_BLOCK": {
        "1": ("oracle", [(c, {"stft_path": (None, 6)}) for c in STFT_CASES if c.startswith("stft")]),
    },
    # the warp kernel's CTA tile and its warp-private tiles share the FFT, the real split (same twiddle table) and the power /
    # magnitude instructions; only the staging of the results differs
    "SYGB200_STFT_CTA_TILE": {
        "1": ("bit", [(c, {"stft_path": (2, 7)}) for c in STFT_CASES if c.startswith("real")]),
    },
    # register-staged warp kernel instead of the TMA ring: the split differs in the last bits; as test_ring_equals_register_staged_kernel
    "SYGB200_RING": {
        "0": (("rtol", 2e-5), [(c, {"stft_path": (1, 2)}) for c in STFT_CASES if c.startswith("ring")]),
    },
}


# ------------------------------------------------------------------------------------------------ inputs (worker and parent)
def fin_many_frames(c, sm_count):
    return 2 * 5 * sm_count * (64 if c["fp"]["mfcc"]["n_mels"] <= 64 else 32)


def feature_input(name, c, sm_count):
    from sygnals_b200.utils import synth
    seed = sum(map(ord, name))
    if c["form"] == "ragged":
        lengths = np.array(c["units"] or [16000, 7000, 300, 11000], dtype=np.int64)
        if c["units"] is None:
            per = sum(1 + int(n) // c["hop"] for n in lengths)
            reps = -(-fin_many_frames(c, sm_count) // per)
            lengths = np.tile(lengths, reps + reps % 2)          # even: the host pipeline's two chunks then split at a repetition
        y = synth.long_signal(int(lengths.sum()), c["sr"], seed=seed).astype(np.float32)
        starts = np.concatenate([[0], np.cumsum(lengths)[:-1]]).astype(np.int64)
        return y, (starts, lengths)
    if c["units"] is None:
        n, L = -(-fin_many_frames(c, sm_count) // (1 + 16000 // c["hop"])), 16000
    else:
        n, L = c["units"]
    y = np.stack([synth.long_signal(L, c["sr"], seed=seed + u).astype(np.float32) * np.float32(10.0 ** (-(u % 3))) for u in range(n)])
    if n > 4:
        y[2] = 0.0
    return y, None


def stft_input(name, c):
    from sygnals_b200.utils import synth
    n, L = c["n"], c["L"]
    buf = np.empty(n * L + 4, dtype=np.float32)                      # 16-byte aligned: the ring kernel's condition
    off = (-buf.ctypes.data // 4) % 4
    y = buf[off:off + n * L].reshape(n, L)
    y[...] = np.stack([synth.mixture(L, 16000, seed=sum(map(ord, name)) + i) for i in range(n)])
    if n > 2:
        y[1] = synth.edge_clip("impulse", L, 16000)
    return y


def welch_input(name, c):
    from sygnals_b200.utils import synth
    sr = 25600
    return np.stack([synth.long_signal(sr, sr, seed=sum(map(ord, name)) + i, block_sec=0.25) for i in range(3)]).astype(np.float32), sr


# ------------------------------------------------------------------------------------------------ worker
def _getters(eng):
    d = eng.lib.dll
    tt, ctas, tiles = eng.lib.last_finalize()
    return np.array([d.syg_debug_last_feature_kernel(), d.syg_debug_last_mel_form(), d.syg_debug_last_features_resident(), tt, ctas,
                     tiles, d.syg_debug_last_stft_path(), d.syg_debug_last_welch_path()], dtype=np.int64)


def run_case(eng, name):
    c = CASES[name]
    res = {}
    if c["kind"] == "features":
        y, rag = feature_input(name, c, eng.sm_count)
        p = _ffi.make_params(eng.lib, c["sr"], c["feats"], c["fl"], c["hop"], feature_params=c["fp"])
        eng.lib.dll.syg_debug_set_resident_min_groups(c["res"])
        try:
            if c["form"] == "ragged":
                out = eng.features_ragged_host(y, eng.ragged_units(rag[0], rag[1], y.size), p)
            elif c["form"] == "vectors":
                out = eng.segment_vectors_host(y.ctypes.data, eng.units_clips(*y.shape), p, [0] * eng.rows(p))
            else:
                out = eng.features_host(y.ravel(), eng.units_clips(*y.shape), p)
        finally:
            eng.lib.dll.syg_debug_set_resident_min_groups(-1)
        res["out"] = out
        res["out:getters"] = _getters(eng)
    elif c["kind"] == "stft":
        y = stft_input(name, c)
        for k in c["kinds"]:
            kind = {"complex": _ffi.OUT_COMPLEX, "magnitude": _ffi.OUT_MAGNITUDE, "power": _ffi.OUT_POWER}[k]
            res[k] = eng.stft_host(y.reshape(-1), eng.units_clips(*y.shape), c["n_fft"], c["hop"], c["n_fft"], 0, True, c["pad"], kind)
            res[k + ":getters"] = _getters(eng)
    else:
        y, sr = welch_input(name, c)
        psd, st = eng.psd_welch_host(y.ravel(), eng.units_clips(*y.shape), sr, 0, c["nperseg"], c["noverlap"], c["nfft"], c["detrend"],
                                     c["scaling"], stats=True)
        res["psd"], res["stats"], res["psd:getters"] = psd, st, _getters(eng)
        res["stats:getters"] = res["psd:getters"]
    return res


def worker_main(backend, out_path, names):
    from backends import get_engine
    eng = get_engine(backend)
    res = {"sm_count": np.array(eng.sm_count)}
    for n in names:
        for k, v in run_case(eng, n).items():
            res[f"{n}/{k}"] = v
    np.savez(out_path, **res)


# ------------------------------------------------------------------------------------------------ parent
ARMS = [(sw, v) for sw, vals in SWITCHES.items() for v in vals]
SWITCH_CASES = [(sw, v, e[0]) for sw, v in ARMS for e in SWITCHES[sw][v][1]]


def child_env(extra):
    env = {k: v for k, v in os.environ.items() if not k.startswith("SYGB200_") or k == "SYGB200_DEVICE"}
    env.update(extra)
    return env


def run_child(backend, out_path, names, extra_env):
    r = subprocess.run([sys.executable, "-s", os.path.abspath(__file__), backend, out_path, ",".join(names)], cwd=ROOT,
                       env=child_env(extra_env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, f"child {extra_env or 'default'} failed:\n{r.stdout[-3000:]}\n{r.stderr[-6000:]}"
    with np.load(out_path) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="module", params=BACKENDS)
def children(request, tmp_path_factory):
    """backend -> {"default": outputs, (switch, value): outputs}: one clean child per arm, all started together."""
    backend = request.param
    if backend == "emu":
        import build_emu
        build_emu.build_emu()                 # once, before any child: concurrent builds would race on the library file
    tmp = tmp_path_factory.mktemp(f"switches_{backend}")
    jobs = {"default": (sorted(CASES), {})}
    for sw, v in ARMS:
        jobs[(sw, v)] = (sorted({e[0] for e in SWITCHES[sw][v][1]}), {sw: v})
    workers = min(len(jobs), os.cpu_count() or 1) if backend == "emu" else 4
    with ThreadPoolExecutor(max_workers=workers) as ex:
        futs = {k: ex.submit(run_child, backend, str(tmp / f"{i}.npz"), names, env) for i, (k, (names, env)) in enumerate(jobs.items())}
        return {k: f.result() for k, f in futs.items()}


def test_switch_table_covers_every_switch_the_library_reads():
    """A new getenv("SYGB200_...") in the library cannot ship without an arm in SWITCHES and an entry in DESIGN.md 6."""
    csrc = os.path.join(ROOT, "sygnals_b200", "csrc")
    read = set()
    for f in sorted(os.listdir(csrc)):
        with open(os.path.join(csrc, f)) as fh:
            read |= set(re.findall(r'getenv\(\s*"(SYGB200_[A-Z0-9_]+)"', fh.read()))
    assert read == set(SWITCHES), f"switches read by the library {sorted(read)} != switches tested here {sorted(SWITCHES)}"
    with open(os.path.join(ROOT, "DESIGN.md")) as fh:
        design = fh.read()
    sec = re.search(r"^## 6\b.*?(?=^## \d)", design, flags=re.S | re.M)
    assert sec, "DESIGN.md has no section 6"
    missing = [s for s in sorted(read) if s not in sec.group(0)]
    assert not missing, f"not documented in DESIGN.md 6: {missing}"


@pytest.mark.parametrize("switch,value,case", SWITCH_CASES, ids=[f"{s[8:]}={v}-{c}" for s, v, c in SWITCH_CASES])
def test_switch_arm(children, switch, value, case):
    base, arm = children["default"], children[(switch, value)]
    relation, entries = SWITCHES[switch][value]
    entry = next(e for e in entries if e[0] == case)
    expect = entry[1]
    relation = entry[2] if len(entry) > 2 else relation          # a case whose arm is the default one (a control) is bit-equal
    keys = sorted(k[len(case) + 1:] for k in arm if k.startswith(case + "/") and not k.endswith(":getters"))
    assert keys, f"no outputs for {case}"
    for key in keys:
        gb, ga = base[f"{case}/{key}:getters"], arm[f"{case}/{key}:getters"]
        for g, (want_default, want_arm) in expect.items():
            i = GETTERS.index(g)
            if want_default != want_arm or want_default is None:
                assert ga[i] != gb[i], f"{key}: switch had no effect ({g} = {ga[i]} in both children)"
            if want_default is not None:
                assert gb[i] == want_default, f"{key}: default child ran {g} = {gb[i]}, expected {want_default}"
            assert ga[i] == want_arm, f"{key}: {switch}={value} ran {g} = {ga[i]}, expected {want_arm}"
        if switch == "SYGB200_FIN_CTAS":
            ctas, tiles = ga[GETTERS.index("fin_ctas")], ga[GETTERS.index("fin_tiles")]
            assert ctas == arm["sm_count"] and tiles > ctas, f"{key}: {ctas} CTAs for {tiles} tiles"
            assert tiles >= 4 * ctas, f"{key}: only {tiles} tiles for {ctas} CTAs"
        a, b = arm[f"{case}/{key}"], base[f"{case}/{key}"]
        assert a.shape == b.shape and a.dtype == b.dtype
        if relation == "bit":
            assert np.array_equal(a, b, equal_nan=True), f"{key}: differs from the default arm on {(a != b).sum()} of {a.size} values"
        elif relation != "oracle":
            bar, x = relation
            scale = np.abs(b).max() if bar == "rtol" else 0.0
            np.testing.assert_allclose(a, b, rtol=x if bar == "rtol" else 0, atol=x if bar == "atol" else 1e-6 * scale)
    check_oracle(case, arm, int(arm["sm_count"]))


# ------------------------------------------------------------------------------------------------ oracle parity
def contrast_ok(y, fl, hop):
    """Frames whose spectral contrast is comparable in FP32: no bin below 1e-5 of the frame's largest (test_parity_cabi.py).  The
    inputs have silent and DC blocks; a DC block's valleys sit at the FP32 noise floor."""
    from oracle import sygnals_oracle as orc
    S = np.abs(orc.compute_stft(np.asarray(y, dtype=np.float64), n_fft=fl, hop_length=hop))
    return S.min(axis=0) >= 1e-5 * S.max(axis=0)


def check_oracle(name, res, sm_count):
    from oracle import sygnals_oracle as orc
    from test_parity_cabi import check_rows, oracle_rows, power_close
    c = CASES[name]
    if c["kind"] == "features":
        y, rag = feature_input(name, c, sm_count)
        sr, fl, hop = c["sr"], c["fl"], c["hop"]
        out = res[f"{name}/out"]
        n_units = len(rag[0]) if rag else y.shape[0]
        units = range(n_units) if n_units <= 12 else range(0, n_units, n_units // 8)
        if c["form"] == "ragged":
            T = [1 + int(n) // hop for n in rag[1]]                  # syg_frame_count, centred frames
            F = np.concatenate([[0], np.cumsum(T)])
            for u in units:
                s, n = rag[0][u], rag[1][u]
                names, ref = oracle_rows(y[s:s + n], sr, c["feats"], fl, hop, c["fp"])
                check_rows(names, out[:, F[u]:F[u + 1]], ref, bin_hz=sr / fl, nyq=sr / 2, contrast_ok=contrast_ok(y[s:s + n], fl, hop))
            return
        for u in units:
            names, ref = oracle_rows(y[u], sr, c["feats"], fl, hop, c["fp"])
            ok = contrast_ok(y[u], fl, hop)
            if c["form"] == "vectors":                             # mean over the unit's frames
                m, r = out[u], ref.mean(axis=1)
                con = np.array([n.startswith("contrast_") for n in names])
                assert not ok.all() or (np.abs(m[con] - r[con]) <= 2e-2).all(), f"unit {u}: contrast means"
                keep = [i for i, n in enumerate(names) if not con[i]]
                check_rows([names[i] for i in keep], m[keep, None], r[keep, None], bin_hz=sr / fl, nyq=sr / 2)
            else:
                check_rows(names, out[u], ref, bin_hz=sr / fl, nyq=sr / 2, contrast_ok=ok)
    elif c["kind"] == "stft":
        y = stft_input(name, c)
        for u in range(c["n"]):
            ref = orc.compute_stft(y[u].astype(np.float64), n_fft=c["n_fft"], hop_length=c["hop"], win_length=c["n_fft"], window="hann",
                                   center=True, pad_mode="reflect" if c["pad"] else "constant")
            P = np.abs(ref) ** 2
            for k in c["kinds"]:
                got = res[f"{name}/{k}"][u]
                assert got.shape == ref.shape
                if k == "complex":
                    scale = np.abs(ref).max(axis=0, keepdims=True)
                    assert (np.abs(got - ref) <= 2e-6 * scale + 1e-12).all(), f"unit {u}: complex output"
                else:
                    power_close(got.astype(np.float64) ** (1 if k == "power" else 2), P)
    else:
        y, sr = welch_input(name, c)
        psd, st = res[f"{name}/psd"], res[f"{name}/stats"]
        for u in range(y.shape[0]):
            x = y[u].astype(np.float64)
            _, ref = orc.compute_psd_welch(x, fs=sr, nperseg=c["nperseg"], noverlap=c["noverlap"], nfft=c["nfft"],
                                           detrend="constant" if c["detrend"] else False, scaling="density" if c["scaling"] == 0 else "spectrum")
            assert psd[u].shape == ref.shape
            assert (np.abs(psd[u] - ref) <= 1e-4 * ref + 1e-6 * ref.max()).all(), f"unit {u}: psd"
            rms = np.sqrt(np.mean(x * x))
            np.testing.assert_allclose(st[u], [rms, np.abs(x).max() / rms, np.abs(x).max()], rtol=1e-5)


if __name__ == "__main__":
    worker_main(sys.argv[1], sys.argv[2], [n for n in sys.argv[3].split(",") if n])
