"""Multi-GPU plumbing of the segment->features path: unit sharding + the one collective of the path.

SURVEY.md 8(e): the path shards over independent units (one unit = one ``extract_features`` call = one clip / segment /
channel-window; the only cross-frame coupling, ``power_to_db(ref=np.max, top_db=80)`` at manager.py:223, is inside a unit).
So there is NO data-path collective: every rank runs the fused kernels on its own contiguous block of units and needs only
its own sample range plus a ``seg_len - seg_hop`` halo (overlapping segments straddle the block edge).  The single exchange
is the final gather of the float32 feature block ``[units, rows, T]`` that feeds the ``sygnals save dataset`` assembly
(``sygnals/cli/save_cmd.py:140-190`` -> ``sygnals/core/ml_utils/formatters.py:51-163``): one
``all_gather_into_tensor`` (NCCL over NVLink/NVSwitch on GPUs; gloo in the CPU tests).

One process per GPU (``torchrun``); nothing here spawns processes.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional, Sequence

import numpy as np

from . import _ffi
from .batch import feature_row_names


def shard_range(n_units: int, rank: int, world: int):
    """Contiguous block partition of ``range(n_units)``: the first ``n_units % world`` ranks own one extra unit."""
    if world < 1 or not 0 <= rank < world:
        raise ValueError(f"rank {rank} / world {world}")
    base, extra = divmod(int(n_units), int(world))
    u0 = rank * base + min(rank, extra)
    return u0, u0 + base + (1 if rank < extra else 0)


@dataclass
class ShardPlan:
    """What one rank needs to run its block of segments of a ``total``-sample recording."""
    rank: int
    world: int
    n_units: int                 # segments of the whole recording
    u0: int                      # this rank owns segments [u0, u1)
    u1: int
    seg_len: int
    seg_hop: int
    sample_begin: int            # this rank needs y[sample_begin:sample_end] (its block plus the halo)
    sample_end: int
    starts: np.ndarray           # int64 [u1-u0]  segment starts relative to sample_begin
    valid: np.ndarray            # int32 [u1-u0]  real samples of each segment (rest is zero padding)
    counts: np.ndarray           # int64 [world]  units per rank (for the gather)

    @property
    def n_local(self) -> int:
        return self.u1 - self.u0


def plan_segments(total_samples: int, sr: int, segment_length_sec: float, overlap_ratio: float = 0.0, pad: bool = True,
                  min_segment_length_sec: Optional[float] = None, rank: int = 0, world: int = 1,
                  lib: Optional[_ffi.Library] = None) -> ShardPlan:
    """Segment table (``segment_fixed_length`` arithmetic, segmentation.py:62-114) cut into per-rank blocks."""
    lib = lib or _ffi.library()
    seg_len, seg_hop, starts, valid = lib.segment_table(total_samples, sr, segment_length_sec, overlap_ratio, pad,
                                                        min_segment_length_sec)
    n = len(starts)
    u0, u1 = shard_range(n, rank, world)
    counts = np.array([shard_range(n, r, world)[1] - shard_range(n, r, world)[0] for r in range(world)], dtype=np.int64)
    if u1 > u0:
        b = int(starts[u0])
        e = int((starts[u0:u1] + valid[u0:u1]).max())
    else:
        b = e = 0
    return ShardPlan(rank, world, n, u0, u1, seg_len, seg_hop, b, e, (starts[u0:u1] - b).astype(np.int64),
                     valid[u0:u1].astype(np.int32), counts)


def _is_torch(x) -> bool:
    return type(x).__module__.startswith("torch")


def _shard_units(eng, plan: ShardPlan, n_have: int, device=None):
    """Unit description of this rank's block relative to its local sample slice.  Regular grids (the usual case: every start is
    ``i * seg_hop`` from the slice's first sample) need no table; irregular ones (``min_segment_length_sec`` dropped a segment) go
    through device / host tables, returned as ``keep`` so the caller holds them for the duration of the call."""
    n = plan.n_local
    regular = n == 0 or bool((plan.starts == np.arange(n, dtype=np.int64) * plan.seg_hop).all())
    if regular:
        return eng.units_clips(n, plan.seg_len, total_len=n_have, stride=plan.seg_hop), None
    if device is not None:
        import torch
        st = torch.from_numpy(plan.starts).to(device)
        va = torch.from_numpy(plan.valid).to(device)
        return eng.units_table(st.data_ptr(), va.data_ptr(), n, plan.seg_len, n_have), (st, va)
    st, va = np.ascontiguousarray(plan.starts), np.ascontiguousarray(plan.valid)
    return eng.units_table(st.ctypes.data, va.ctypes.data, n, plan.seg_len, n_have), (st, va)


def run_shard(y_local, plan: ShardPlan, sr: int, features: Sequence[str], frame_length: int = 2048, hop_length: int = 512,
              center: bool = True, window: str = "hann", feature_params: Optional[dict] = None,
              engine: Optional[_ffi.Engine] = None, aggregation=None, out=None):
    """Features of this rank's segments.  ``y_local`` holds ``y[plan.sample_begin:plan.sample_end]`` (numpy: host path;
    CUDA torch tensor: device path, asynchronous on the current stream).  Returns float32 ``[n_local, rows, T]``, or -- with
    ``aggregation`` ('mean' | 'std' | 'median' | 'min' | 'max' or a per-feature dict: format_feature_vectors_per_segment,
    formatters.py:51-163, every segment one row) -- float64 ``[n_local, rows]`` straight from the fused device path
    (``syg_segment_vectors_f32``: the frame features never leave the library's workspace).  ``out``: optional preallocated result."""
    n_have = int(y_local.shape[0])
    if n_have != plan.sample_end - plan.sample_begin:
        raise ValueError(f"y_local has {n_have} samples, the shard needs {plan.sample_end - plan.sample_begin}")
    ids = None
    if aggregation is not None:
        from .core.ml_utils.formatters import _agg_ids
        ids = _agg_ids(feature_row_names(features, feature_params), aggregation)
    if _is_torch(y_local) and y_local.is_cuda:
        import torch
        eng = engine or _ffi.engine(y_local.device.index or 0)
        p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
        rows, T = eng.rows(p), eng.frame_count(plan.seg_len, frame_length, hop_length, center)
        shape = (plan.n_local, rows) if ids is not None else (plan.n_local, rows, T)
        if out is None:
            out = torch.empty(shape, dtype=torch.float64 if ids is not None else torch.float32, device=y_local.device)
        if out.numel():
            units, keep = _shard_units(eng, plan, n_have, y_local.device)
            y32 = y_local if (y_local.dtype == torch.float32 and y_local.is_contiguous()) else y_local.contiguous().float()
            stream = torch.cuda.current_stream(y_local.device).cuda_stream
            if ids is not None:
                eng.segment_vectors_dev(y32.data_ptr(), units, p, ids, out.data_ptr(), stream)
            else:
                eng.features_dev(y32.data_ptr(), units, p, out.data_ptr(), stream)
            # `keep` / `y32` may be released now: the kernels are queued on the CURRENT torch stream and the caching allocator hands
            # a freed block only to work queued later on that same stream, so no host synchronisation is needed here
            del keep
        return out
    eng = engine or _ffi.engine()
    p = _ffi.reference_params(eng.lib, sr, list(features), frame_length, hop_length, center, window, feature_params)
    y32 = np.ascontiguousarray(y_local, dtype=np.float32)
    units, keep = _shard_units(eng, plan, n_have, None)
    if ids is not None:
        return eng.segment_vectors_host(y32.ctypes.data, units, p, ids)
    return eng.features_host(y32, units, p)


def gather_features(local, plan: ShardPlan, group=None):
    """The path's one collective: every rank contributes ``[n_local, rows, T]`` and receives ``[n_units, rows, T]`` in
    segment order.  Ranks own different unit counts (block partition), so blocks are padded to the largest count for one
    ``all_gather_into_tensor`` and trimmed afterwards.  torch tensors in, torch tensor out (CUDA -> NCCL, CPU -> gloo);
    numpy in -> numpy out through a CPU tensor."""
    import torch
    import torch.distributed as dist
    was_numpy = not _is_torch(local)
    t = torch.from_numpy(np.ascontiguousarray(local)) if was_numpy else local.contiguous()
    if plan.world == 1 or not (dist.is_available() and dist.is_initialized()):
        return local
    rows_T = tuple(t.shape[1:])
    mx = int(plan.counts.max())
    padded = t
    if t.shape[0] != mx:
        padded = torch.zeros((mx,) + rows_T, dtype=t.dtype, device=t.device)
        padded[: t.shape[0]] = t
    buf = torch.empty((plan.world * mx,) + rows_T, dtype=t.dtype, device=t.device)
    dist.all_gather_into_tensor(buf, padded, group=group)
    if int(plan.counts.min()) == mx:
        full = buf
    else:
        full = torch.cat([buf[r * mx: r * mx + int(c)] for r, c in enumerate(plan.counts)], dim=0)
    return full.numpy() if was_numpy else full


def segment_features_sharded(y, sr: int, segment_length_sec: float, features: Sequence[str], overlap_ratio: float = 0.0,
                             pad: bool = True, min_segment_length_sec: Optional[float] = None, frame_length: int = 2048,
                             hop_length: int = 512, center: bool = True, window: str = "hann",
                             feature_params: Optional[dict] = None, rank: Optional[int] = None, world: Optional[int] = None,
                             gather: bool = True, group=None, engine: Optional[_ffi.Engine] = None,
                             aggregation=None) -> Dict[str, object]:
    """``batch.segment_features`` over ``world`` ranks: each rank slices its sample range (block + halo) out of ``y`` (every
    rank is handed the same recording, or at least its own range of it), runs the fused kernels on its block of segments and
    -- if ``gather`` -- takes part in the final all-gather.  ``aggregation`` ('mean' | 'std' | 'median' | 'min' | 'max' or a
    per-feature dict) reduces every segment's frames on the device first.  Returns {'names', 'features', 'plan'}."""
    if rank is None or world is None:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(group), dist.get_world_size(group)
        else:
            rank, world = 0, 1
    lib = engine.lib if engine is not None else None
    plan = plan_segments(int(y.shape[0]), sr, segment_length_sec, overlap_ratio, pad, min_segment_length_sec, rank, world, lib)
    # aggregation: format_feature_vectors_per_segment (formatters.py:51-163) on the device BEFORE the gather, so the collective
    # carries [segments, rows] float64 instead of [segments, rows, T] float32
    local = run_shard(y[plan.sample_begin:plan.sample_end], plan, sr, features, frame_length, hop_length, center, window,
                      feature_params, engine, aggregation=aggregation)
    names = feature_row_names(features, feature_params)
    out = gather_features(local, plan, group) if gather else local
    return {"names": names, "features": out, "plan": plan}
