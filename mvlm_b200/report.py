"""Per-landmark consensus report: which landmarks of a scan to trust, and why (DESIGN.md 7h).

`Pipeline.predict_*(..., report=True)` and `sharding.predict_mesh_view_split(..., report=True)` return one
LandmarkReport per scan.  The consensus fields come from the report kernel (`ops.consensus(report=True)`); the surface
fields are computed here from the triangle each landmark was snapped to, in torch fp64 on the device.  A pass's report
travels to the host as one byte row per scan (`pack` / `unpack`), so it costs one page-locked copy.
"""
from __future__ import annotations

import dataclasses

import numpy as np
import torch

__all__ = ["LandmarkReport", "STATUS_NAMES"]

STATUS_NAMES = ("ransac", "all_lines", "few_lines")


@dataclasses.dataclass
class LandmarkReport:
    """One scan.  L landmarks, V views; points in the scan's own coordinates (pre-alignment undone).

    landmarks        (L,3) f64    the landmarks the call returns
    error            float        the call's last_error
    status           (L,) int8    0 ransac: a hypothesis was accepted; 1 all_lines: >= 3 lines, none accepted, LSQ over
                                  all kept lines; 2 few_lines: < 3 lines, plain LSQ (0 lines: the point 0)
    n_lines          (L,) int32   lines kept by the heat-value filter
    n_inliers        (L,) int32   lines of the final fit: status 0 the winning hypothesis's inliers, else n_lines
    inliers          (L,V) bool   view v's line is one of them (views the filter removed: False)
    consensus_points (L,3) f64    the consensus point before snapping
    rms              (L,) f64     sqrt(mean squared distance of those lines to the consensus point); NaN without lines
    covariance       (L,3,3) f64  sigma^2 J^-1, J = sum (I - n n^T), sigma^2 = sum d^2 / (2k - 3) over the k lines of the
                                  fit; NaN when k < 2 or J is singular
    surface_distance (L,) f64     |snapped landmark - consensus point|
    triangle         (L,) int32   the triangle the landmark was snapped to
    barycentric      (L,3) f64    of the snapped point in that triangle
    nearest_vertex   (L,) int32   the triangle's corner with the largest barycentric weight (ties: the first corner)
    peaks            (L,V,3) f32  the per-view (row, col, value) peaks the rays were built from
    """
    landmarks: np.ndarray
    error: float
    status: np.ndarray
    n_lines: np.ndarray
    n_inliers: np.ndarray
    inliers: np.ndarray
    consensus_points: np.ndarray
    rms: np.ndarray
    covariance: np.ndarray
    surface_distance: np.ndarray
    triangle: np.ndarray
    barycentric: np.ndarray
    nearest_vertex: np.ndarray
    peaks: np.ndarray

    def save(self, path) -> None:
        """Every field into one .npz file (np.load(path) gives them back by name)."""
        np.savez(path, **{f.name: getattr(self, f.name) for f in dataclasses.fields(self)})


# Fields computed on the device and their per-scan shapes, largest item first so that every field of a packed row
# starts aligned to its item size.
def _layout(l: int, v: int):
    return (("consensus_points", np.float64, (l, 3)), ("rms", np.float64, (l,)), ("covariance", np.float64, (l, 3, 3)),
            ("surface_distance", np.float64, (l,)), ("barycentric", np.float64, (l, 3)),
            ("n_lines", np.int32, (l,)), ("n_inliers", np.int32, (l,)), ("triangle", np.int32, (l,)),
            ("nearest_vertex", np.int32, (l,)), ("peaks", np.float32, (l, v, 3)),
            ("status", np.int8, (l,)), ("inliers", np.bool_, (l, v)))


_TORCH = {np.float64: torch.float64, np.int32: torch.int32, np.float32: torch.float32, np.int8: torch.int8,
          np.bool_: torch.bool}


def barycentric(points: torch.Tensor, corners: torch.Tensor) -> torch.Tensor:
    """(N,3) points and (N,3,3) triangle corners (fp64) -> (N,3) barycentric coordinates of each point's projection on
    its triangle's plane."""
    a, b, c = corners[:, 0], corners[:, 1], corners[:, 2]
    v0, v1, v2 = b - a, c - a, points - a
    d00, d01, d11 = (v0 * v0).sum(1), (v0 * v1).sum(1), (v1 * v1).sum(1)
    d20, d21 = (v2 * v0).sum(1), (v2 * v1).sum(1)
    den = d00 * d11 - d01 * d01
    wb = (d11 * d20 - d01 * d21) / den
    wc = (d00 * d21 - d01 * d20) / den
    return torch.stack([1.0 - wb - wc, wb, wc], dim=1)


def pack(consensus_points, n_lines, rep, snapped, tri, meshes, peaks) -> torch.Tensor:
    """Device fields of the S scans of a pass -> (S, bytes) uint8 on the device, one row per scan.
    consensus_points (S,L,3), n_lines (S,L), rep the (S,L,...) ops.ConsensusReport, snapped (S,L,3), tri (S,L),
    meshes S (verts (Nv,3) f32, tris (Nt,3) i32) device pairs, peaks (L,S*V,3) f32."""
    s, l = tri.shape
    bary, nearest = [], []
    for i, (verts, tris) in enumerate(meshes):
        idx = tris[tri[i].long()].long()                      # (L,3) corner vertex ids
        b = barycentric(snapped[i], verts[idx].double())
        bary.append(b)
        nearest.append(idx.gather(1, b.argmax(1, keepdim=True))[:, 0].int())  # argmax: first maximum
    v = peaks.shape[1] // s
    fields = {"consensus_points": consensus_points, "rms": rep.rms, "covariance": rep.covariance,
              "surface_distance": torch.linalg.vector_norm(snapped - consensus_points, dim=2),
              "barycentric": torch.stack(bary), "n_lines": n_lines, "n_inliers": rep.n_inliers, "triangle": tri,
              "nearest_vertex": torch.stack(nearest), "peaks": peaks.reshape(l, s, v, 3).transpose(0, 1),
              "status": rep.status, "inliers": rep.inliers}
    cols = []
    for name, dtype, _ in _layout(l, v):
        t = fields[name].contiguous().reshape(s, -1)
        assert t.dtype == _TORCH[dtype], (name, t.dtype)
        cols.append(t.view(torch.uint8))
    row = torch.cat(cols, dim=1)
    pad = -row.shape[1] % 8
    return torch.nn.functional.pad(row, (0, pad)) if pad else row


def unpack(row: np.ndarray, n_views: int, landmarks: np.ndarray, error: float) -> LandmarkReport:
    """One scan's packed row (host uint8) -> LandmarkReport with the given landmarks and error."""
    l = landmarks.shape[0]
    out, off = {}, 0
    for name, dtype, shape in _layout(l, n_views):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        out[name] = row[off:off + n].view(dtype).reshape(shape).copy()
        off += n
    return LandmarkReport(landmarks=landmarks, error=error, **out)


def map_back(rep: LandmarkReport, a: np.ndarray, b: np.ndarray) -> LandmarkReport:
    """Report of a pre-aligned scan (p' = A p + b, A = scale * rotation) in the scan's own coordinates: points through
    prealign.invert, the covariance to A^-1 C A^-T, rms and surface_distance divided by the scale |det A|^(1/3).  The
    counts, status, inlier mask, triangle, barycentric coordinates and peaks do not change."""
    from .utils import prealign

    ainv = np.linalg.inv(a)
    scale = abs(np.linalg.det(a)) ** (1.0 / 3.0)
    return dataclasses.replace(rep, landmarks=prealign.invert(rep.landmarks, a, b),
                               consensus_points=prealign.invert(rep.consensus_points, a, b),
                               covariance=ainv @ rep.covariance @ ainv.T, rms=rep.rms / scale,
                               surface_distance=rep.surface_distance / scale)
