"""The per-landmark consensus report (DESIGN.md 7h) on the GPU: the report kernel against the numpy restatement in
report_ref.py, the report leaving landmarks, errors and launches alone, and the report of every pipeline entry point
and of the view-split path."""
import dataclasses
import os

import numpy as np
import pytest
import torch

from mvlm_b200 import ops, report, synth
from mvlm_b200.io_obj import Mesh
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.pipeline import general_pipeline as gp
from mvlm_b200.utils import prealign
from mvlm_b200.weights import seeded_state_dict

import report_ref

pytestmark = pytest.mark.gpu

DEV = "cuda"


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _rays(n_scans, l, v, seed):
    rays = [synth.synthetic_rays(l, v, outlier_frac=0.3, seed=seed + i) for i in range(n_scans)]
    return tuple(np.concatenate([r[k] for r in rays], axis=1) for k in range(3))


def _check_slot(got, ref, where):
    """got: this slot's kernel outputs; ref: report_ref.slot_report."""
    assert ref["margin"] > 1e-9, (f"{where}: a line's squared distance lies within 1e-9 (relative) of the inlier "
                                  f"threshold in the restatement, so an fp64 rounding difference could flip it; this "
                                  f"slot cannot be compared exactly (margin {ref['margin']:.3g})")
    assert got["status"] == ref["status"], where
    assert got["n_lines"] == ref["n_lines"] and got["n_inliers"] == ref["n_inliers"], where
    assert np.array_equal(got["inliers"], ref["inliers"]), where
    if ref["n_lines"] == 0:
        assert np.isnan(got["rms"]) and np.array_equal(got["point"], np.zeros(3)), where
    elif ref["n_inliers"] == 1:  # the LSQ point of one line lies on it: both distances are rounding noise
        assert got["rms"] < 1e-9 and ref["rms"] < 1e-9, where
    else:
        assert abs(got["rms"] - ref["rms"]) <= 1e-9 * ref["rms"], (where, got["rms"], ref["rms"])
        assert np.abs(got["point"] - ref["point"]).max() <= 1e-8, where
    assert np.array_equal(np.isnan(got["covariance"]), np.isnan(ref["covariance"])), where
    if np.isfinite(ref["covariance"]).all():
        scale = np.abs(ref["covariance"]).max()
        assert np.abs(got["covariance"] - ref["covariance"]).max() <= 1e-9 * scale, where


def _run(peaks, starts, ends, draws, n_scans, **kw):
    """Consensus without and with the report, and the library launches of each."""
    torch.cuda.synchronize()
    lib = ops._lib.load()
    lib.mvlm_launch_count(1)
    plain = ops.consensus_multiscan(t(peaks), t(starts), t(ends), draws, n_scans, **kw)
    n_plain = lib.mvlm_launch_count(1)
    with_report = ops.consensus_multiscan(t(peaks), t(starts), t(ends), draws, n_scans, report=True, **kw)
    n_report = lib.mvlm_launch_count(1)
    assert (n_plain, n_report) == (3, 4)
    for a, b in zip(plain, with_report[:3]):  # the report leaves landmarks, errors and line counts alone
        assert torch.equal(a, b)
    host = lambda x: x.cpu().numpy()  # noqa: E731
    return tuple(map(host, with_report[:3])), ops.ConsensusReport(*map(host, with_report[3]))


def _check_pass(peaks, starts, ends, tables, per_scan, slots, mode, **kw):
    n_scans, v = len(tables), peaks.shape[1] // len(tables)
    draws = t(np.stack(tables).view(np.int32)) if per_scan else t(tables[0].view(np.int32))
    (lm, err, nl), rep = _run(peaks, starts, ends, draws, n_scans, mode=mode, **kw)
    assert rep.status.dtype == np.int8 and rep.inliers.dtype == np.bool_ and rep.covariance.shape[-2:] == (3, 3)
    # status 0: rms^2 sums the squared distances the hypothesis kernel scored, to the refit point it kept, in its
    # order, so sqrt(error) matches bit for bit -- the report kernel's refit point is out_landmarks
    s0 = rep.status == 0
    assert np.array_equal(rep.rms[s0], np.sqrt(err[s0]))
    assert (err[rep.status == 1] == report_ref.NO_FIT).all() and (err[rep.status == 2] == 0).all()
    assert np.array_equal(rep.n_inliers[~s0], nl[~s0])
    for s, l in slots:
        sl = slice(s * v, (s + 1) * v)
        ref = report_ref.slot_report(peaks[l, sl, 2], starts[l, sl], ends[l, sl], tables[s][l], mode=mode, **kw)
        got = {"status": rep.status[s, l], "n_lines": nl[s, l], "n_inliers": rep.n_inliers[s, l],
               "inliers": rep.inliers[s, l], "point": lm[s, l], "rms": rep.rms[s, l],
               "covariance": rep.covariance[s, l]}
        _check_slot(got, ref, (mode, s, l))
    return rep


@pytest.mark.parametrize("mode", ["quantile", "absolute"])
@pytest.mark.parametrize("n_hyp", [1, 16384])
@pytest.mark.parametrize("per_scan_draws", [False, True])
def test_report_kernel_matches_restatement(lib, mode, n_hyp, per_scan_draws):
    """C5-style rays (84 landmarks x 200 views, 30 % outliers), a pass of 3 scans.  At H = 16384 the numpy restatement
    (a few thousand hypotheses per second) checks one landmark per scan, at H = 1 every landmark."""
    n_scans, l, v = 3, 84, 200
    peaks, starts, ends = _rays(n_scans, l, v, 300)
    tables = [synth.hypothesis_table(l, n_hyp, seed=11 + (i if per_scan_draws else 0)) for i in range(n_scans)]
    slots = [(s, i) for s in range(n_scans) for i in range(l)] if n_hyp == 1 else \
        [(s, (29 * s + 7) % l) for s in range(n_scans)]
    rep = _check_pass(peaks, starts, ends, tables, per_scan_draws, slots, mode, threshold_absolute=0.5)
    if n_hyp == 1:  # one hypothesis is often rejected: both RANSAC outcomes are exercised
        assert {0, 1} <= set(np.unique(rep.status).tolist())
    else:
        assert (rep.status == 0).all()


@pytest.mark.parametrize("mode", ["quantile", "absolute"])
def test_report_edge_cases(lib, mode):
    """0, 1 and 2 kept lines, all-equal heat values (the median filter keeps none) and a NaN heat value, in a pass of
    two scans."""
    n_scans, l, v = 2, 8, 12
    peaks, starts, ends = _rays(n_scans, l, v, 500)
    vals = np.tile(np.linspace(0.05, 0.95, v, dtype=np.float32), (l, n_scans))
    if mode == "absolute":
        for i, k in enumerate((0, 1, 2)):      # scan 0, landmarks 0-2: keep k lines
            vals[i, :v] = np.where(np.arange(v) < k, 0.9, 0.1)
        vals[3, v - 1] = np.nan                  # a NaN value fails `>`: that line is dropped
        vals[4, v:v + 2] = 0.9                   # scan 1: 2 lines
        vals[4, v + 2:] = 0.1
    else:
        vals[0, :v] = 0.5                        # all equal: nothing above the median
        vals[1, v + 3] = np.nan                  # np.quantile -> NaN: no line kept
        vals[2, :v] = np.where(np.arange(v) < 2, 0.9, 0.1)  # median 0.1: 2 lines
    peaks[..., 2] = vals
    tables = [synth.hypothesis_table(l, 64, seed=3)] * n_scans
    rep = _check_pass(peaks, starts, ends, tables, False, [(s, i) for s in range(n_scans) for i in range(l)], mode,
                      threshold_absolute=0.5)
    if mode == "absolute":
        assert rep.status[0, :3].tolist() == [2, 2, 2] and rep.n_inliers[0, :3].tolist() == [0, 1, 2]
        assert np.isnan(rep.rms[0, 0]) and np.isnan(rep.covariance[0, :2]).all()
        assert np.isfinite(rep.covariance[0, 2]).all() and not rep.inliers[0, 3, v - 1]
        assert rep.status[1, 4] == 2 and rep.n_inliers[1, 4] == 2
    else:
        assert rep.status[0, 0] == 2 and rep.n_inliers[0, 0] == 0 and not rep.inliers[0, 0].any()
        assert rep.status[1, 1] == 2 and rep.n_inliers[1, 1] == 0
        assert rep.n_inliers[0, 2] == 2 and np.isfinite(rep.covariance[0, 2]).all()


# --------------------------------------------------------------------------------------------------------------------
# pipeline entry points
# --------------------------------------------------------------------------------------------------------------------
SD = seeded_state_dict(73, "RGB+depth", 1234)


def _scan(grid, seed, tex=True):
    v, uv, tr = synth.face_mesh(grid=grid, seed=seed)
    return Mesh(verts=v, tris=tr, uvs=uv, texture=synth.face_texture(128, seed=seed) if tex else None)


def _meshes():
    return [_scan(60, 11), _scan(80, 12), _scan(50, 13, False), _scan(70, 14)]


def _pipeline(n_views=8, seed=5, **kw):
    return create_pipeline("dtu3d", n_views=n_views, weights=SD, seed=seed, n_hypotheses=4, verbose=False,
                           image_size=(128, 128), **kw)


def _same_report(a, b, where=""):
    assert (a is None) == (b is None), where
    if a is None:
        return
    for f in dataclasses.fields(a):
        x, y = getattr(a, f.name), getattr(b, f.name)
        if f.name == "error":
            assert x == y, where
        else:
            assert x.dtype == y.dtype and x.shape == y.shape, (where, f.name)
            assert np.array_equal(x, y, equal_nan=x.dtype.kind == "f"), (where, f.name)


def test_pipeline_report_equals_plain_result(lib):
    dm = _pipeline()
    mesh = _meshes()[0]
    dm.predict_mesh(mesh, report=True)  # plans, graphs and pinned buffers of both forms exist after these two calls
    lm = dm.predict_mesh(mesh)
    err = dm.last_error
    torch.cuda.synchronize()
    lib.mvlm_launch_count(1)
    assert np.array_equal(dm.predict_mesh(mesh), lm)
    off = lib.mvlm_launch_count(1)
    r = dm.predict_mesh(mesh, report=True)
    on = lib.mvlm_launch_count(1)
    assert on == off + 1
    assert isinstance(r, report.LandmarkReport)
    assert np.array_equal(r.landmarks, lm) and r.error == err == dm.last_error
    l, v = lm.shape[0], 8
    assert r.inliers.shape == (l, v) and r.peaks.shape == (l, v, 3) and r.covariance.shape == (l, 3, 3)
    assert np.array_equal(r.n_inliers[r.status != 0], r.n_lines[r.status != 0])
    assert np.array_equal(r.inliers.sum(1), r.n_inliers)
    # the surface fields: barycentrics reproduce the snapped point, distances and nearest corners follow from them
    corners = mesh.verts[mesh.tris[r.triangle]].astype(np.float64)
    assert np.abs(np.einsum("lk,lkc->lc", r.barycentric, corners) - lm).max() <= 1e-9 * mesh.bbox_diagonal
    assert np.allclose(r.surface_distance, np.linalg.norm(lm - r.consensus_points, axis=1), rtol=1e-12, atol=0)
    assert np.array_equal(r.nearest_vertex, mesh.tris[r.triangle][np.arange(l), np.argmax(r.barycentric, axis=1)])


@pytest.mark.parametrize("seed", [5, None])
def test_predict_meshes_reports_equal_one_scan_at_a_time(lib, monkeypatch, seed):
    monkeypatch.setattr(gp, "PASS_PIXELS", 3 * 8 * 128 * 128)
    dm = _pipeline(seed=seed)
    assert dm._scans_per_pass() == 3
    meshes = _meshes()
    batch = [meshes[0], None, *meshes[1:]]
    np.random.seed(77)
    ref = [None if m is None else dm.predict_mesh(m, report=True) for m in batch]
    state = np.random.get_state()
    np.random.seed(77)
    got = dm.predict_meshes(batch, report=True)
    after = np.random.get_state()
    assert after[0] == state[0] and np.array_equal(after[1], state[1]) and after[2:] == state[2:]
    assert len(got) == len(ref)
    for i, (a, b) in enumerate(zip(got, ref)):
        _same_report(a, b, i)
    assert dm.last_error == ref[-1].error
    if seed is not None:  # one pass of 3 scans: exactly one launch more with the report
        dm.predict_meshes(meshes[:3])
        torch.cuda.synchronize()
        lib.mvlm_launch_count(1)
        dm.predict_meshes(meshes[:3])
        off = lib.mvlm_launch_count(1)
        dm.predict_meshes(meshes[:3], report=True)
        assert lib.mvlm_launch_count(1) == off + 1


def test_predict_files_and_folder_reports(lib, monkeypatch, tmp_path):
    monkeypatch.setattr(gp, "PASS_PIXELS", 3 * 8 * 128 * 128)
    paths = []
    for i, m in enumerate(_meshes()):
        paths.append(synth.write_obj(tmp_path / f"s{i}.obj", m.verts, m.uvs, m.tris, m.texture))
    dm = _pipeline()
    ref = [dm.predict_one_file(p, report=True) for p in paths]
    got = dm.predict_files([paths[0], tmp_path / "missing.obj", *paths[1:]], report=True)
    for i, (a, b) in enumerate(zip(got, [ref[0], None, *ref[1:]])):
        _same_report(a, b, i)
    out = dm.predict_folder(tmp_path, out=tmp_path / "lm", report=True)
    for p, r in zip(paths, ref):
        _same_report(out[p], r, p.name)
        assert np.array_equal(np.loadtxt(tmp_path / "lm" / f"{p.stem}_dtu3d.txt", delimiter=","), r.landmarks)
        with np.load(tmp_path / "lm" / f"{p.stem}_dtu3d_report.npz") as z:
            assert np.array_equal(z["landmarks"], r.landmarks) and np.array_equal(z["inliers"], r.inliers)
            assert float(z["error"]) == r.error


def test_pre_align_report_is_the_aligned_scans_report_mapped_back(lib):
    cfg = {"align_center_of_mass": True, "rot_x": 10, "rot_y": -20, "rot_z": 5, "scale": 1.1}
    tr = synth.random_view_transforms(8, seed=4)
    mesh = _meshes()[1]
    a, b = prealign.affine(mesh.verts, cfg)
    aligned = dataclasses.replace(mesh, verts=prealign.apply(mesh.verts, a, b))
    plain = _pipeline(transforms=tr).predict_mesh(aligned, report=True)
    dm = _pipeline(transforms=tr, pre_align=cfg)
    got = dm.predict_mesh(mesh, report=True)
    _same_report(got, report.map_back(plain, a, b))
    assert np.array_equal(got.landmarks, dm.predict_mesh(mesh))
    assert np.allclose(got.rms, plain.rms / 1.1, rtol=1e-12, equal_nan=True)


def test_seam_path_rejects_report(lib, tmp_path):
    m = _meshes()[0]
    path = synth.write_obj(tmp_path / "s.obj", m.verts, m.uvs, m.tris, m.texture)
    dm = _pipeline(render_image_stack=True, render_image_folder=tmp_path)
    with pytest.raises(ValueError, match="fused device path"):
        dm.predict_one_file(path, report=True)


def test_view_split_report_equals_single_gpu_report(lib):
    import torch.distributed as dist

    from mvlm_b200.sharding import predict_mesh_view_split

    mesh = _scan(60, 2)
    tr = synth.random_view_transforms(6, seed=2)
    dm = _pipeline(n_views=6, seed=3, transforms=tr)
    single = dm.predict_mesh(mesh, report=True)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29534")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        split = predict_mesh_view_split(dm, mesh, tr, report=True)
        plain = predict_mesh_view_split(dm, mesh, tr)
    finally:
        if created:
            dist.destroy_process_group()
    _same_report(split, single)
    assert np.array_equal(plain, single.landmarks) and dm.last_error == single.error
