"""Multi-GPU host logic: one process per GPU (torch.distributed), no collective on the data path
when scans are sharded; one all-gather of the per-view peaks when ONE scan's views are split.

The reference has no distributed code (only an optional in-process DataParallel wrap,
src/mvlm/prediction/paulsenpredictor.py:104-105); scans are independent units and views of a scan
are independent up to the peak stage (the quantile filter needs all views, estimator3d.py:140-147),
which fixes where the exchange has to sit (SURVEY.md 8e).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist


def shard_scans(n_scans: int, rank: int, world: int) -> list[int]:
    """Static round-robin assignment of scan indices to ranks."""
    return list(range(rank, n_scans, world))


def split_views(n_views: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous (start, count) block of views for `rank`; the first n_views % world ranks get one more."""
    base, rem = divmod(n_views, world)
    count = base + (1 if rank < rem else 0)
    start = rank * base + min(rank, rem)
    return start, count


def _view_rows(n_views: int, world: int, device) -> torch.Tensor:
    """Row of global view v in a gather buffer of `world` slots of ceil(n_views / world) views (rank-major)."""
    slot = split_views(n_views, 0, world)[1]
    rows = []
    for r in range(world):
        s, c = split_views(n_views, r, world)
        rows.extend(r * slot + i for i in range(c))
    return torch.tensor(rows, dtype=torch.long, device=device)


_ROWS_CACHE: dict = {}


def allgather_peaks(local_peaks: torch.Tensor, n_views: int, group=None) -> torch.Tensor:
    """local_peaks (L, V_local, 3) float32 of this rank's view block -> (L, V, 3) on every rank.

    Fallback of the view-split path (non-default peak selection, sliced plans; the default path gathers the arg-max
    KEYS in place, see allgather_keys).  One in-place collective of L*ceil(V/world)*12 bytes per rank (25 KB at L=84,
    V=200, world=8): latency-bound; NCCL over NVLink on GPUs, gloo on CPU (tests).  The block is written view-major into
    this rank's slot of the receive buffer, the gather runs in place, and ONE indexed read (cached row table) puts the
    views in order: no zero-filled send buffer, no per-rank copy loop."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    l = local_peaks.shape[0]
    slot = split_views(n_views, 0, world)[1]
    start, count = split_views(n_views, rank, world)
    assert local_peaks.shape[1] == count, (local_peaks.shape, count)
    recv = torch.empty((world, slot, l, 3), dtype=local_peaks.dtype, device=local_peaks.device)
    if count < slot:
        recv[rank, count:].zero_()  # the unused row of a short block travels too: keep it defined
    recv[rank, :count].copy_(local_peaks.permute(1, 0, 2))
    dist.all_gather_into_tensor(recv.view(-1), recv[rank].reshape(-1), group=group)
    key = (n_views, world, str(local_peaks.device))
    if key not in _ROWS_CACHE:
        _ROWS_CACHE[key] = _view_rows(n_views, world, local_peaks.device)
    return recv.view(world * slot, l, 3).index_select(0, _ROWS_CACHE[key]).permute(1, 0, 2).contiguous()


def allgather_keys(keys_all: torch.Tensor, group=None) -> None:
    """In-place all-gather of the arg-max keys: keys_all (world, slot_views, L) int64, slot [rank] already written by
    this rank's network (Hourglass.forward_keys).  One NCCL collective, no staging copy."""
    rank = dist.get_rank(group)
    dist.all_gather_into_tensor(keys_all.view(-1), keys_all[rank].reshape(-1), group=group)


# Scans at least this large take the sharded upload in predict_mesh_view_split.  Measured (profiles/r1_view_split_c4.txt):
# 5 MB scan 1.05 -> 0.37 ms on 8 GPUs, 0.55 -> 0.53 ms on 2; 47 MB scan 8.98 -> 1.20 ms on 8, 3.40 -> 2.95 ms on 2.
SHARDED_UPLOAD_MIN_BYTES = 4 << 20


def allgather_bytes(array: np.ndarray, device, stage=None, name: str = "a", group=None) -> torch.Tensor:
    """`array` is the same on every rank: rank r moves only the r-th 1/world of its bytes from host to device and the
    slices are all-gathered (NCCL over NVLink on GPUs, gloo on CPU), so a scan crosses each rank's PCIe link and host
    memory once per `world` ranks instead of once per rank.  Returns the whole array on `device`."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    a = np.ascontiguousarray(array)
    raw = a.reshape(-1).view(np.uint8)
    chunk = (-(-raw.size // world) + 15) // 16 * 16
    lo, hi = min(rank * chunk, raw.size), min((rank + 1) * chunk, raw.size)
    send = torch.zeros((chunk,), dtype=torch.uint8, device=device) if hi - lo < chunk else \
        torch.empty((chunk,), dtype=torch.uint8, device=device)
    if hi > lo:
        part = raw[lo:hi]
        if stage is not None and torch.device(device).type == "cuda":
            send[:hi - lo].copy_(stage.stage(name + "@shard", part), non_blocking=True)
        else:
            send[:hi - lo].copy_(torch.from_numpy(part.copy()))
    recv = torch.empty((world * chunk,), dtype=torch.uint8, device=device)
    dist.all_gather_into_tensor(recv, send, group=group)
    return recv[:raw.size].view(torch.from_numpy(a[:0].reshape(-1).copy()).dtype).view(a.shape)


def upload_mesh_sharded(renderer, mesh, group=None):
    """DeviceMesh of a scan every rank holds in host memory, each rank uploading 1/world of it (allgather_bytes)."""
    from .utils.render3d import DeviceMesh, _on_current_stream, _PinnedStage

    device = renderer.device
    stage = None
    if torch.device(device).type == "cuda":
        ring = renderer.__dict__.setdefault("_shard_stages", [_PinnedStage() for _ in range(2)])
        renderer._shard_i = getattr(renderer, "_shard_i", 0) + 1
        stage = ring[renderer._shard_i % len(ring)]
        if stage.done is not None:
            stage.done.synchronize()  # the slot's previous transfer has left the host buffers
    arrays = {name: _on_current_stream(a, ready) if isinstance(a, torch.Tensor)  # on the device already
              else allgather_bytes(a, device, stage, name, group) for name, a, ready in mesh.arrays()}
    if stage is not None:
        stage.done = torch.cuda.Event()
        stage.done.record()
    return DeviceMesh.from_device(mesh, arrays)


def _mesh_bytes(mesh) -> int:
    """Bytes of the scan's host arrays (Mesh.arrays), the upload that upload_mesh_sharded splits over the ranks; for a
    scan with texture pages this includes their 12-byte-per-page table."""
    return sum(a.nbytes for _, a, _ in mesh.arrays() if isinstance(a, np.ndarray))


def predict_mesh_view_split(pipeline, mesh, transforms: np.ndarray, group=None) -> np.ndarray:
    """One scan whose views are split over the ranks of `group` (BASELINE.json config 4):
    every rank holds the whole mesh (uploaded in `world` slices and all-gathered when it is large), rasterises and runs
    the CNN on its block of views, the peaks are all-gathered, and every rank finishes rays / consensus / snap redundantly (it is microseconds of
    work and removes a broadcast of the result)."""
    from . import ops

    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    r, p, e = pipeline.renderer_3d, pipeline.predictor_2d, pipeline.estimator_3d
    transforms = np.asarray(transforms)
    n_views = transforms.shape[0]
    start, count = split_views(n_views, rank, world)
    slot = split_views(n_views, 0, world)[1]
    size = r.image_size
    n_lm = p.get_lm_count()
    # every rank needs the whole mesh: large scans are uploaded 1/world per rank and all-gathered over NVLink
    dmesh = upload_mesh_sharded(r, mesh, group) if world > 1 and _mesh_bytes(mesh) >= SHARDED_UPLOAD_MIN_BYTES else r.upload(mesh)
    dev = dmesh.verts.device
    # more ranks than views: the ranks without a view skip raster and CNN and still join the collectives
    local = r.render_device(dmesh, transforms[start:start + count]) if count > 0 else None
    if p.can_write_keys(max(count, 1), size[0], size[1]):
        # default path: the last convolution's fused arg-max writes this rank's keys straight into its slot of the
        # (persistent) gather buffer, ONE in-place collective, ONE kernel from the gathered keys to the peaks of all views
        kb = pipeline.__dict__.get("_vs_keys")
        if kb is None or kb.shape != (world, slot, n_lm) or kb.device != dev:
            kb = pipeline.__dict__["_vs_keys"] = torch.zeros((world, slot, n_lm), dtype=torch.int64, device=dev)
        if count > 0:
            p.predict_keys_device(local["u8"], kb[rank, :count])
        allgather_keys(kb, group)
        peaks = ops.peaks_from_gathered_keys(kb, n_views, size[1])
    else:
        peaks_local = p.predict_landmarks_device(local["u8"]) if count > 0 else \
            torch.empty((n_lm, 0, 3), dtype=torch.float32, device=dev)
        peaks = allgather_peaks(peaks_local, n_views, group)
    if e.seed is None:
        raise ValueError("view-split prediction needs a seeded hypothesis table (Estimator3D.seed)")
    # rotation matrices of ALL views and the hypothesis table are cached on the device across scans
    if getattr(pipeline, "_vs_rot_key", None) != transforms.tobytes():
        from .utils.render3d import rotation_matrices

        pipeline._vs_rot = torch.from_numpy(rotation_matrices(transforms).reshape(-1, 9)).to(peaks.device)
        pipeline._vs_rot_key = transforms.tobytes()
    starts, ends = e.estimate_landmark_lines_device(peaks, transforms, r.image_size[0], rot=pipeline._vs_rot)
    draws = e.seeded_draws_device(peaks.shape[0])
    lm, err, _ = e.estimate_landmarks_from_lines_device(peaks, starts, ends, draws)
    snapped, _ = ops.snap_to_mesh(dmesh.verts, dmesh.tris, lm, grid=dmesh.snap_grid())
    pipeline.last_error = float((err.sum() / err.numel()).item())
    return snapped.cpu().numpy()


def predict_files(pipeline, paths, group=None):
    """Batch driver (reference main.py:50-62 is a serial loop): scans are dealt round-robin to the
    ranks; rank 0 receives all results.  Returns {index: (L,3) array} on rank 0, own share elsewhere."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    idx = shard_scans(len(paths), rank, world)
    mine = dict(zip(idx, pipeline.predict_files([paths[i] for i in idx])))  # prefetching loader, see Pipeline.predict_files
    if world == 1:
        return mine
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=group)
    if rank != 0:
        return mine
    out = {}
    for d in gathered:
        out.update(d)
    return out
