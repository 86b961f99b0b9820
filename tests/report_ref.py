"""numpy restatement of the per-landmark consensus report (DESIGN.md 7h), built on the oracle's consensus stages.

slot_report() gives one (landmark, scan) slot's consensus fields from its peaks, rays and raw hypothesis draws.  It
follows oracle.stages.landmarks_from_lines (filter, RANSAC over the hypothesis list, first strict minimum, fallbacks)
and keeps what that function drops: the winner's inlier set and the lines and point of the final fit.
"""
import numpy as np

from oracle import stages

NO_FIT = 100000000  # estimator3d.py:95


def covariance(pa: np.ndarray, pb: np.ndarray, point: np.ndarray) -> np.ndarray:
    """sigma^2 J^-1 of the LSQ point of lines (pa, pb): J = sum (I - n n^T), sigma^2 = sum d^2 / (2k - 3).  NaN when
    k < 2 or J has an eigenvalue at or below 1e-15 times the largest (np.linalg.pinv's cut-off)."""
    k = len(pa)
    if k < 2:
        return np.full((3, 3), np.nan)
    n = (pb - pa) / np.linalg.norm(pb - pa, axis=1)[:, None]
    j = k * np.eye(3) - n.T @ n
    lam, vec = np.linalg.eigh(j)
    if np.abs(lam).min() <= 1e-15 * np.abs(lam).max():
        return np.full((3, 3), np.nan)
    s2 = stages.point_line_sqdist(point, pa, pb).sum() / (2 * k - 3)
    return s2 * (vec / lam) @ vec.T


def slot_report(values, starts, ends, raw_draws, mode="quantile", threshold_quantile=0.5, threshold_absolute=0.5,
                dist_thres=100.0) -> dict:
    """values (V,) f32 heat values, starts / ends (V,3) f64, raw_draws (H,8) u32.  Returns status, n_lines, n_inliers,
    inliers (V,) bool, point (3,), rms, covariance (3,3) and `margin`: the smallest |d^2 - dist_thres| / dist_thres
    over the inlier tests of every hypothesis, so a caller can tell when an fp64 rounding difference could flip an
    inlier decision."""
    keep = stages.line_filter_mask(np.asarray(values, np.float32), mode, threshold_quantile, threshold_absolute)
    views = np.nonzero(keep)[0]
    pa, pb = starts[keep], ends[keep]
    n = len(pa)
    used = np.ones(n, bool)
    margin = np.inf
    status = 2 if n < 3 else 1
    if n == 0:
        point = np.zeros(3)
    else:
        point = stages.lsq_intersection(pa, pb)
    if n >= 3:
        best = NO_FIT
        for ran in stages.hypotheses_for(raw_draws, n):
            dist = stages.point_line_sqdist(stages.lsq_intersection(pa[ran], pb[ran]), pa, pb)
            inl = dist < dist_thres
            margin = min(margin, float(np.min(np.abs(dist - dist_thres))) / dist_thres)
            if inl.sum() > n / 3:
                p = stages.lsq_intersection(pa[inl], pb[inl])
                err = stages.point_line_sqdist(p, pa[inl], pb[inl]).sum() / inl.sum()
                if err < best:
                    best, point, used, status = err, p, inl, 0
    inliers = np.zeros(len(values), bool)
    inliers[views[used]] = True
    k = int(used.sum())
    d2 = stages.point_line_sqdist(point, pa[used], pb[used]) if k else np.zeros(0)
    return {"status": status, "n_lines": n, "n_inliers": k, "inliers": inliers, "point": point,
            "rms": np.sqrt(d2.sum() / k) if k else np.nan, "covariance": covariance(pa[used], pb[used], point),
            "margin": margin}
