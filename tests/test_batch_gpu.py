"""Several scans per device pass: the multi-scan raster, consensus and snap, and the batch drivers built on them, must
give every scan exactly (bit for bit) what one scan at a time gives it."""
import numpy as np
import pytest
import torch

from mvlm_b200 import ops, synth
from mvlm_b200.io_obj import Mesh
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.pipeline import general_pipeline as gp
from mvlm_b200.utils.render3d import rotation_matrices
from mvlm_b200.weights import seeded_state_dict

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _scan(grid, seed, tex="rgb"):
    v, uv, t = synth.face_mesh(grid=grid, seed=seed)
    texture = None if tex is None else synth.face_texture(128, seed=seed)
    if tex == "rgba":
        texture = np.concatenate([texture, np.full(texture.shape[:2] + (1,), 200, np.uint8)], axis=2)
    return Mesh(verts=v, tris=t, uvs=uv, texture=texture)


def _dev(mesh):
    up = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    return up(mesh.verts), (up(mesh.uvs) if mesh.texture is not None else None), up(mesh.tris), up(mesh.texture)


def _rot(n_views, seed):
    return torch.from_numpy(rotation_matrices(synth.random_view_transforms(n_views, seed=seed)).reshape(-1, 9)).to(DEV)


@pytest.mark.parametrize("mode", list(ops.CHANNEL_MODES))
def test_raster_multiscan_equals_per_scan(lib, mode):
    scans = [_dev(_scan(40, 1, "rgb")), _dev(_scan(90, 2, "rgba")), _dev(_scan(60, 3, None))]
    v, h, w = 5, 96, 128
    rots = [_rot(v, 10 + i) for i in range(len(scans))]
    got = ops.raster_multiscan(scans, torch.cat(rots), h, w, mode, want_f32=True, want_tri=True, want_z=True)
    for i, (s, r) in enumerate(zip(scans, rots)):
        ref = ops.raster_multiview(*s, r, h, w, mode, want_f32=True, want_tri=True, want_z=True)
        for k in ("u8", "f32", "tri", "z"):
            assert torch.equal(got[k][i * v:(i + 1) * v], ref[k]), (mode, i, k)


def test_raster_multiscan_chunked_path(lib):
    # a million-vertex scan: 16 MB of transformed vertices per view, so the 24 views of the pass run in chunks of 16
    # (scan, view) pairs that straddle the scans
    scans = [_dev(_scan(70, 4, "rgb")), _dev(_scan(1001, 5, "rgb")), _dev(_scan(50, 6, None))]
    v, h, w = 8, 64, 64
    assert lib.mvlm_raster_multiscan_workspace_bytes(3, v, h, w, 1001 * 1001) < 3 * v * (h * w * 8 + 1001 * 1001 * 16)
    rots = [_rot(v, 20 + i) for i in range(3)]
    got = ops.raster_multiscan(scans, torch.cat(rots), h, w, want_tri=True, want_z=True)
    for i, (s, r) in enumerate(zip(scans, rots)):
        ref = ops.raster_multiview(*s, r, h, w, want_tri=True, want_z=True)
        for k in ("u8", "tri", "z"):
            assert torch.equal(got[k][i * v:(i + 1) * v], ref[k]), (i, k)


@pytest.mark.parametrize("mode", ["quantile", "absolute"])
@pytest.mark.parametrize("n_hyp", [1, 16384])
@pytest.mark.parametrize("per_scan_draws", [False, True])
def test_consensus_multiscan_equals_per_scan(lib, mode, n_hyp, per_scan_draws):
    n_scans, l, v = 5, 73, 8
    rays = [synth.synthetic_rays(l, v, outlier_frac=0.3, seed=100 + i) for i in range(n_scans)]
    peaks = np.concatenate([r[0] for r in rays], axis=1)
    starts = np.concatenate([r[1] for r in rays], axis=1)
    ends = np.concatenate([r[2] for r in rays], axis=1)
    if mode == "absolute":
        peaks[..., 2] = np.where(np.arange(n_scans * v) % 3 == 0, 0.1, 0.9)  # some landmarks keep < 3 lines
        peaks[::7, : 3 * v, 2] = 0.0
    tables = [synth.hypothesis_table(l, n_hyp, seed=7 + (i if per_scan_draws else 0)) for i in range(n_scans)]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(DEV)  # noqa: E731
    draws = t(np.stack(tables).view(np.int32)) if per_scan_draws else t(tables[0].view(np.int32))
    kw = dict(mode=mode, threshold_absolute=0.5)
    lm, err, nl = ops.consensus_multiscan(t(peaks), t(starts), t(ends), draws, n_scans, **kw)
    for i in range(n_scans):
        sl = slice(i * v, (i + 1) * v)
        r_lm, r_err, r_nl = ops.consensus(t(peaks[:, sl]), t(starts[:, sl]), t(ends[:, sl]), t(tables[i].view(np.int32)),
                                          **kw)
        assert torch.equal(lm[i], r_lm) and torch.equal(err[i], r_err) and torch.equal(nl[i], r_nl), i


def test_snap_to_meshes_equals_per_scan(lib):
    meshes = [_scan(30, 1), _scan(310, 2), _scan(80, 3), _scan(120, 4)]
    assert meshes[1].tris.shape[0] >= ops.SNAP_GRID_MIN_TRIS > max(m.tris.shape[0] for m in meshes if m is not meshes[1])
    dev = [_dev(m) for m in meshes]
    rng = np.random.RandomState(3)
    lms = []
    for m in meshes:  # near the surface, and a few far away (the grid query hands those to the scan kernel)
        pts = m.verts[rng.randint(0, m.verts.shape[0], 73)].astype(np.float64) + rng.normal(0, 2.0, (73, 3))
        pts[:3] += 400.0
        lms.append(pts)
    lm = torch.from_numpy(np.stack(lms)).to(DEV)
    table = []
    for i, d in enumerate(dev):
        grid = ops.SnapGrid(d[0], d[2]) if d[2].shape[0] >= ops.SNAP_GRID_MIN_TRIS else None
        if grid is not None:  # the far landmarks really are handed back to the batched scan kernel (shells == -1)
            _, _, stats = grid.query(lm[i].contiguous(), want_stats=True)
            assert (stats[:3, 1] == -1).all() and (stats[3:, 1] >= 0).any()
        table.append((d[0], d[2], grid))
    pts, tid = ops.snap_to_meshes(table, lm)
    for i, (verts, tris, grid) in enumerate(table):
        ref_p, ref_t = ops.snap_to_mesh(verts, tris, lm[i].contiguous(), grid=grid)
        assert torch.equal(pts[i], ref_p) and torch.equal(tid[i], ref_t), i
        brute_p, brute_t = ops.snap_to_mesh(verts, tris, lm[i].contiguous())
        assert torch.equal(pts[i], brute_p) and torch.equal(tid[i], brute_t), i
    # one scan with a grid goes through the grid query's own launches
    one_p, one_t = ops.snap_to_meshes(table[1:2], lm[1:2].contiguous())
    assert torch.equal(one_p[0], pts[1]) and torch.equal(one_t[0], tid[1])


# --------------------------------------------------------------------------------------------------------------------
# batch drivers
# --------------------------------------------------------------------------------------------------------------------
SD = seeded_state_dict(73, "RGB+depth", 1234)


def _meshes():
    return [_scan(60, 11), _scan(80, 12, "rgba"), _scan(50, 13, None), _scan(70, 14), _scan(60, 15), _scan(90, 16),
            _scan(40, 17)]


def _pipeline(n_views=8, seed=5, **kw):
    return create_pipeline("dtu3d", n_views=n_views, weights=SD, seed=seed, n_hypotheses=4, verbose=False,
                           image_size=(128, 128), **kw)


def _three_per_pass(monkeypatch):
    monkeypatch.setattr(gp, "PASS_PIXELS", 3 * 8 * 128 * 128)


def _same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert (x is None) == (y is None)
        if x is not None:
            assert np.array_equal(x, y)


@pytest.mark.parametrize("n_views,seed", [(8, 5), (8, None), (6, 5), (6, None)])
@pytest.mark.parametrize("depth", [1, 2])
def test_predict_meshes_equals_one_scan_at_a_time(lib, monkeypatch, n_views, seed, depth):
    _three_per_pass(monkeypatch)
    dm = _pipeline(n_views, seed)
    expected = 1 if (n_views != 8 and seed is None) else (3 if n_views == 8 else 4)
    assert dm._scans_per_pass() == expected
    meshes = _meshes()
    batch = [meshes[0], None, *meshes[1:4], None, *meshes[4:]]  # 7 scans: passes of 3, 3 and a tail of 1 at 8 views
    np.random.seed(77)
    ref, errs = [], []
    for m in batch:
        ref.append(None if m is None else dm.predict_mesh(m))
        errs.append(dm.last_error)
    state = np.random.get_state()
    np.random.seed(77)
    got = dm.predict_meshes(batch, depth=depth)
    _same(got, ref)
    assert dm.last_error == errs[-1]
    after = np.random.get_state()
    assert after[0] == state[0] and np.array_equal(after[1], state[1]) and after[2:] == state[2:]


def test_predict_meshes_pre_align(lib, monkeypatch):
    _three_per_pass(monkeypatch)
    dm = _pipeline(pre_align={"align_center_of_mass": True, "rot_x": 10, "rot_y": -20, "rot_z": 5, "scale": 1.1})
    meshes = _meshes()[:5]
    _same(dm.predict_meshes(meshes), [dm.predict_mesh(m) for m in meshes])


@pytest.mark.parametrize("parser", ["host", "gpu"])
def test_predict_files_and_folder_equal_one_file_at_a_time(lib, monkeypatch, tmp_path, parser):
    _three_per_pass(monkeypatch)
    paths = []
    for i, m in enumerate(_meshes()[:5]):
        tex = m.texture[..., :3] if m.texture is not None else None
        paths.append(synth.write_obj(tmp_path / f"s{i}.obj", m.verts, m.uvs, m.tris, tex))
    dm = _pipeline(obj_parser=parser)
    ref = [dm.predict_one_file(p) for p in paths]
    files = [paths[0], tmp_path / "missing.obj", *paths[1:]]
    _same(dm.predict_files(files), [ref[0], None, *ref[1:]])
    out = dm.predict_folder(tmp_path, out=tmp_path / "lm")
    _same([out[p] for p in sorted(paths)], [ref[paths.index(p)] for p in sorted(paths)])


def test_one_pass_launches_what_one_scan_launches(lib, monkeypatch):
    _three_per_pass(monkeypatch)
    dm = _pipeline()
    meshes = _meshes()[:3]
    dm.predict_meshes(meshes)  # plans, graphs and buffers of both pass sizes exist after these two calls
    dm.predict_mesh(meshes[0])
    torch.cuda.synchronize()
    lib.mvlm_launch_count(1)
    dm.predict_mesh(meshes[0])
    single = lib.mvlm_launch_count(1)
    dm.predict_meshes(meshes)
    batched = lib.mvlm_launch_count(1)
    assert single > 100 and batched == single
