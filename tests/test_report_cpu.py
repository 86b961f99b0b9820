"""The per-landmark consensus report (DESIGN.md 7h) on the CPU: the numpy restatement in report_ref.py against
geometry with a known answer, and the host side of mvlm_b200.report (packing, barycentric coordinates, the pre-align
mapping of every field)."""
import numpy as np
import pytest
import torch

from mvlm_b200 import report
from mvlm_b200.ops import ConsensusReport
from mvlm_b200.utils import prealign

import report_ref


def _lines_through(x, dirs, offsets):
    """Lines along unit `dirs` through x + offsets, the offsets (k,2) taken across each line."""
    starts, ends = [], []
    for d, (e1, e2) in zip(dirs, offsets):
        u = np.cross(d, [0.0, 0.0, 1.0] if abs(d[2]) < 0.9 else [1.0, 0.0, 0.0])
        u /= np.linalg.norm(u)
        w = np.cross(d, u)
        c = x + e1 * u + e2 * w
        starts.append(c - 300.0 * d)
        ends.append(c + 300.0 * d)
    return np.array(starts), np.array(ends)


def _dirs(rng, k):
    d = rng.normal(size=(k, 3))
    return d / np.linalg.norm(d, axis=1)[:, None]


def _draws(h, seed=0):
    return np.random.RandomState(seed).randint(0, 2 ** 32, (h, 8), dtype=np.uint64).astype(np.uint32)


def _report(starts, ends, values=None, h=64, **kw):
    values = np.full(len(starts), 0.9, np.float32) if values is None else np.asarray(values, np.float32)
    return report_ref.slot_report(values, starts, ends, _draws(h), mode="absolute", threshold_absolute=0.5, **kw)


def test_concurrent_lines_have_zero_rms():
    rng = np.random.RandomState(1)
    x = np.array([10.0, -20.0, 30.0])
    s, e = _lines_through(x, _dirs(rng, 10), np.zeros((10, 2)))
    r = _report(s, e)
    assert r["status"] == 0 and r["n_inliers"] == 10 and r["inliers"].all()
    assert r["rms"] < 1e-10 and np.abs(r["point"] - x).max() < 1e-10
    assert np.isfinite(r["covariance"]).all() and np.abs(r["covariance"]).max() < 1e-18


def test_every_status():
    rng = np.random.RandomState(2)
    x = np.array([5.0, 6.0, -7.0])
    # RANSAC accepts: 12 lines through x (0.3 mm across), 4 outliers 60 mm off; the mask is exactly the 12
    s, e = _lines_through(x, _dirs(rng, 16), np.r_[rng.normal(0, 0.3, (12, 2)), np.full((4, 2), 60.0)])
    r = _report(s, e)
    assert (r["status"], r["n_lines"], r["n_inliers"]) == (0, 16, 12)
    assert np.array_equal(r["inliers"], np.arange(16) < 12)
    # the view mask is in view order: views the filter removed are False, the kept ones map back to their views
    vals = np.where(np.arange(16) % 2 == 0, 0.9, 0.1)
    r = _report(s, e, vals)
    assert r["n_lines"] == 8 and np.array_equal(r["inliers"], (np.arange(16) % 2 == 0) & (np.arange(16) < 12))
    # no accepted hypothesis: 9 lines 200 mm apart; LSQ over all of them, rms is the true value, not 1e8
    s9, e9 = _lines_through(np.zeros(3), _dirs(rng, 9), rng.uniform(-200, 200, (9, 2)))
    r = _report(s9, e9)
    assert (r["status"], r["n_lines"], r["n_inliers"]) == (1, 9, 9) and r["inliers"].all()
    d2 = ((np.cross(r["point"] - s9, r["point"] - e9) ** 2).sum(1)) / ((e9 - s9) ** 2).sum(1)
    assert 10.0 < r["rms"] < 1e4 and abs(r["rms"] - np.sqrt(d2.mean())) <= 1e-12 * r["rms"]
    # fewer than 3 lines: 0, 1 and 2 kept
    for k in (0, 1, 2):
        r = _report(s, e, np.where(np.arange(16) < k, 0.9, 0.1))
        assert (r["status"], r["n_lines"], r["n_inliers"]) == (2, k, k)
        assert np.array_equal(r["inliers"], np.arange(16) < k)
        if k == 0:
            assert np.isnan(r["rms"]) and np.array_equal(r["point"], np.zeros(3))
        else:
            assert np.isfinite(r["rms"])
        assert np.isnan(r["covariance"]).all() == (k < 2)
    # two skew lines: 2k - 3 = 1 degree of freedom, J full rank
    assert np.isfinite(_report(s, e, np.where(np.arange(16) < 2, 0.9, 0.1))["covariance"]).all()


def test_parallel_lines_give_nan_covariance():
    d = np.array([[0.0, 0.6, 0.8]] * 6)
    s, e = _lines_through(np.array([1.0, 2.0, 3.0]), d, np.random.RandomState(3).normal(0, 1.0, (6, 2)))
    r = _report(s, e)
    assert r["n_inliers"] == 6 and np.isfinite(r["rms"]) and np.isnan(r["covariance"]).all()


def test_covariance_matches_monte_carlo():
    """Rays through a point, each displaced across its direction by N(0, sigma^2) per axis.  Over T trials the LSQ
    estimates scatter with covariance sigma^2 J^-1; the predicted covariance (averaged over the trials) must match the
    empirical one.  Whitened by the prediction, the empirical covariance has eigenvalues 1 +- O(sqrt(2/T)) = 1 +- 0.022
    at T = 4000; the bar is 0.12 (5.4 standard deviations).  The mean sigma^2 estimate is unbiased with 2k - 3 degrees
    of freedom (relative standard deviation sqrt(2/9)/sqrt(T) = 0.0075 at k = 6); its bar is 0.04.  A divisor of 2k
    instead of 2k - 3 would be off by 25 %."""
    rng = np.random.RandomState(4)
    x, k, sigma, trials = np.array([3.0, -4.0, 12.0]), 6, 0.5, 4000
    dirs = _dirs(rng, k)
    est, covs, s2 = [], [], []
    for _ in range(trials):
        s, e = _lines_through(x, dirs, rng.normal(0, sigma, (k, 2)))
        p = report_ref.stages.lsq_intersection(s, e)
        c = report_ref.covariance(s, e, p)
        est.append(p)
        covs.append(c)
        s2.append(report_ref.stages.point_line_sqdist(p, s, e).sum() / (2 * k - 3))
    emp = np.cov(np.array(est).T)
    pred = np.mean(covs, axis=0)
    chol = np.linalg.cholesky(pred)
    white = np.linalg.solve(chol, np.linalg.solve(chol, emp).T)
    lam = np.linalg.eigvalsh(white)
    assert np.abs(lam - 1).max() < 0.12, lam
    assert abs(np.mean(s2) / sigma ** 2 - 1) < 0.04
    assert (np.abs(np.mean(est, axis=0) - x) < 5 * np.sqrt(np.diag(pred) / trials)).all()  # unbiased


def test_pre_align_maps_the_consensus_fields_back():
    """The report of lines moved into a pre-aligned frame (p' = A p + b, A = 1.1 R), mapped back by the report's own
    mapping, equals the report of the original lines."""
    rng = np.random.RandomState(5)
    x = np.array([20.0, 10.0, -5.0])
    # outliers so far off that only the all-inlier hypotheses are accepted: both frames pick the same inlier set
    s, e = _lines_through(x, _dirs(rng, 14), np.r_[rng.normal(0, 0.5, (10, 2)), np.full((4, 2), 3000.0)])
    a, b = prealign.affine(rng.normal(0, 30, (50, 3)), {"align_center_of_mass": True, "rot_x": 10, "rot_y": -20,
                                                         "rot_z": 5, "scale": 1.1})
    plain = _report(s, e, h=256)
    moved = _report(s @ a.T + b, e @ a.T + b, h=256)
    assert plain["status"] == 0 and plain["n_inliers"] == 10
    for key in ("status", "n_lines", "n_inliers"):
        assert plain[key] == moved[key]
    assert np.array_equal(plain["inliers"], moved["inliers"])
    ainv = np.linalg.inv(a)
    assert np.allclose(prealign.invert(moved["point"][None], a, b)[0], plain["point"], rtol=0, atol=1e-9)
    assert abs(moved["rms"] / 1.1 - plain["rms"]) <= 1e-9 * plain["rms"]
    assert np.allclose(ainv @ moved["covariance"] @ ainv.T, plain["covariance"], rtol=1e-7,
                       atol=1e-9 * np.abs(plain["covariance"]).max())


def _packed_scan(l=5, v=4, seed=6):
    """A one-scan pass on the CPU: a two-triangle mesh, snapped points on it, arbitrary consensus fields."""
    rng = np.random.RandomState(seed)
    verts = torch.tensor([[0, 0, 0], [2, 0, 0], [0, 2, 0], [2, 2, 1]], dtype=torch.float32)
    tris = torch.tensor([[0, 1, 2], [1, 3, 2]], dtype=torch.int32)
    tri = torch.tensor([[0, 0, 1, 1, 0][:l]], dtype=torch.int32)
    bary = np.array([[0.5, 0.5, 0.0], [0.2, 0.3, 0.5], [0.1, 0.8, 0.1], [1 / 3, 1 / 3, 1 / 3], [0.0, 0.25, 0.75]])[:l]
    corners = verts[tris[tri[0].long()].long()].double().numpy()
    snapped = torch.from_numpy(np.einsum("lk,lkc->lc", bary, corners))[None]
    cp = snapped + torch.from_numpy(rng.normal(0, 1, (1, l, 3)))
    cov = rng.normal(size=(l, 3, 3))
    rep = ConsensusReport(status=torch.tensor([[0, 1, 2, 0, 0][:l]], dtype=torch.int8),
                          n_inliers=torch.arange(l, dtype=torch.int32)[None],
                          inliers=torch.from_numpy(rng.uniform(size=(1, l, v)) > 0.5),
                          rms=torch.from_numpy(rng.uniform(size=(1, l))),
                          covariance=torch.from_numpy(cov @ cov.transpose(0, 2, 1))[None])
    peaks = torch.from_numpy(rng.uniform(size=(l, v, 3)).astype(np.float32))
    nl = torch.full((1, l), v, dtype=torch.int32)
    row = report.pack(cp, nl, rep, snapped, tri, [(verts, tris)], peaks)
    assert row.dtype == torch.uint8 and row.shape[0] == 1 and row.shape[1] % 8 == 0
    lm = snapped[0].numpy()
    return report.unpack(row[0].numpy(), v, lm, 1.5), dict(cp=cp[0].numpy(), rep=rep, peaks=peaks.numpy(),
                                                              bary=bary, lm=lm, tris=tris.numpy(), tri=tri[0].numpy())


def test_pack_unpack_and_surface_fields():
    r, src = _packed_scan()
    assert r.error == 1.5 and r.landmarks is src["lm"]
    assert np.array_equal(r.consensus_points, src["cp"])
    assert np.array_equal(r.status, src["rep"].status[0].numpy()) and r.status.dtype == np.int8
    assert np.array_equal(r.inliers, src["rep"].inliers[0].numpy()) and r.inliers.dtype == np.bool_
    assert np.array_equal(r.covariance, src["rep"].covariance[0].numpy()) and r.covariance.shape == (5, 3, 3)
    assert np.array_equal(r.peaks, src["peaks"]) and r.peaks.dtype == np.float32
    assert np.array_equal(r.n_lines, np.full(5, 4)) and np.array_equal(r.triangle, src["tri"])
    assert np.allclose(r.barycentric, src["bary"], rtol=0, atol=1e-12)
    assert np.allclose(r.surface_distance, np.linalg.norm(r.consensus_points - r.landmarks, axis=1), rtol=1e-15)
    # the corner with the largest weight; the exact tie (0.5, 0.5, 0) of landmark 0 goes to the first corner
    corners = src["tris"][src["tri"]]
    assert np.array_equal(r.nearest_vertex, corners[np.arange(5), np.argmax(src["bary"], axis=1)])
    assert r.nearest_vertex[0] == corners[0, 0]


def test_map_back_maps_each_field(tmp_path):
    r, _ = _packed_scan()
    a, b = prealign.affine(np.random.RandomState(7).normal(0, 30, (20, 3)),
                           {"align_center_of_mass": True, "rot_x": 30, "rot_y": 10, "rot_z": -40, "scale": 0.8})
    m = report.map_back(r, a, b)
    ainv = np.linalg.inv(a)
    assert np.array_equal(m.landmarks, prealign.invert(r.landmarks, a, b))
    assert np.array_equal(m.consensus_points, prealign.invert(r.consensus_points, a, b))
    assert np.allclose(m.covariance, np.einsum("ij,ljk,mk->lim", ainv, r.covariance, ainv), rtol=1e-12, atol=0)
    assert np.allclose(m.rms, r.rms / 0.8, rtol=1e-14) and np.allclose(m.surface_distance, r.surface_distance / 0.8,
                                                                        rtol=1e-14)
    for key in ("status", "n_lines", "n_inliers", "inliers", "triangle", "barycentric", "nearest_vertex", "peaks"):
        assert np.array_equal(getattr(m, key), getattr(r, key)), key
    assert m.error == r.error
    r.save(tmp_path / "r.npz")
    with np.load(tmp_path / "r.npz") as z:
        assert set(z.files) == {f for f in r.__dataclass_fields__}
        assert np.array_equal(z["covariance"], r.covariance) and float(z["error"]) == r.error


def test_exported():
    import mvlm
    import mvlm_b200

    assert mvlm.LandmarkReport is mvlm_b200.LandmarkReport is report.LandmarkReport


@pytest.mark.parametrize("mode", ["quantile", "absolute"])
def test_nan_and_equal_heat_values_keep_no_line(mode):
    s, e = _lines_through(np.zeros(3), _dirs(np.random.RandomState(8), 6), np.zeros((6, 2)))
    vals = np.full(6, 0.9 if mode == "absolute" else 0.7, np.float32)
    if mode == "absolute":
        vals[2] = np.nan
        r = report_ref.slot_report(vals, s, e, _draws(4), mode=mode)
        assert r["n_lines"] == 5 and not r["inliers"][2]
    else:
        r = report_ref.slot_report(vals, s, e, _draws(4), mode=mode)   # all equal: nothing above the median
        assert r["n_lines"] == 0 and r["status"] == 2 and np.isnan(r["rms"])
        vals[1] = np.nan
        assert report_ref.slot_report(vals, s, e, _draws(4), mode=mode)["n_lines"] == 0
