"""PLY / STL scans on the GPU: the device decoder and weld (csrc/mesh_parse.cu) against the host loader, vertex-colour
rasterisation against the numpy rule on the C oracle's triangle ids, and the pipeline's scan_formats."""
import numpy as np
import pytest
import torch

import mesh_ref
from mvlm_b200 import ops, synth
from mvlm_b200.io_mesh import load_mesh, load_ply_stl
from mvlm_b200.io_obj import Mesh, load_obj
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.pipeline import general_pipeline as gp
from mvlm_b200.utils.render3d import rotation_matrices
from mvlm_b200.weights import seeded_state_dict
from oracle import native, stages

pytestmark = pytest.mark.gpu

DEV = "cuda"
FORMATS = ("obj", "ply", "stl")


def _np(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _same(a, b):
    a, b = _np(a), _np(b)
    assert (a is None) == (b is None)
    if a is not None:
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _decode_equals_host(path, on_device=True):
    g = load_ply_stl(path, parser="gpu")
    h = load_ply_stl(path, parser="host")
    assert isinstance(g.verts, torch.Tensor) == on_device
    if on_device:
        g.geometry_ready.synchronize()
    _same(g.verts, h.verts)
    _same(g.tris, h.tris)
    _same(g.colors, h.colors)
    return g, h


@pytest.fixture(scope="module")
def face():
    v, uv, t = synth.face_mesh(grid=90, seed=5)
    rng = np.random.RandomState(9)
    return v, uv, t, rng.randint(0, 256, (len(v), 3)).astype(np.uint8)


@pytest.mark.parametrize("fmt", ["binary_little_endian", "binary_big_endian"])
@pytest.mark.parametrize("pos_type", ["float", "double"])
@pytest.mark.parametrize("with_colors", [False, True])
def test_device_ply_equals_host(lib, tmp_path, face, fmt, pos_type, with_colors):
    v, _, t, c = face
    p = synth.write_ply(tmp_path / "s.ply", v, t, c if with_colors else None, fmt=fmt, pos_type=pos_type,
                        count_type="uchar", index_type="uint")
    _decode_equals_host(p)


def test_device_stl_equals_host(lib, tmp_path, face):
    v, _, t, _ = face
    g, h = _decode_equals_host(synth.write_stl(tmp_path / "s.stl", v, t, header=b"solid header of a binary file"))
    _same(h.verts, mesh_ref.read_stl(tmp_path / "s.stl")[0])
    nan = float("nan")
    soup = np.array([[-0.0, 0, 0], [1, 0, 0], [0, 1, 0], [0.0, 0, 0], [1, 0, 0], [0, 1, 0], [nan, 0, 0], [1, 0, 0],
                     [nan, 0, 0], [1, 0, 0], [0, 1, 0], [1, 0, 0], [2, 2, 2], [2, 2, 2], [2, 2, 2]], np.float32)
    synth.write_stl(tmp_path / "w.stl", soup, np.arange(15).reshape(5, 3))
    _decode_equals_host(tmp_path / "w.stl")


def test_device_decode_at_config4_size(lib, tmp_path):
    v, _, t = synth.face_mesh(grid=1001, seed=3)  # 2M triangles
    assert len(t) == 2_000_000
    c = (np.arange(len(v) * 3) % 251).astype(np.uint8).reshape(-1, 3)
    _decode_equals_host(synth.write_stl(tmp_path / "big.stl", v, t))
    _decode_equals_host(synth.write_ply(tmp_path / "big.ply", v, t, c, fmt="binary_big_endian"))


def test_fallbacks_return_the_host_arrays(lib, tmp_path, face):
    v, _, t, c = face
    quads = [list(t[0]) + [7]] + [list(x) for x in t[1:]]
    _decode_equals_host(synth.write_ply(tmp_path / "q.ply", v, quads, c), on_device=False)
    _decode_equals_host(synth.write_ply(tmp_path / "a.ply", v, t, c, fmt="ascii"), on_device=False)
    _decode_equals_host(synth.write_stl(tmp_path / "a.stl", v, t, binary=False), on_device=False)
    bad = synth.write_ply(tmp_path / "r.ply", v, [[0, 1, len(v)]] + [list(x) for x in t[1:]])
    with pytest.raises(ValueError, match=f"face references vertex {len(v)} of {len(v)}"):
        load_ply_stl(bad, parser="gpu")
    hdr = tmp_path / "h.ply"
    hdr.write_bytes(b"ply\nformat binary_middle_endian 1.0\nend_header\n")
    with pytest.raises(ValueError, match="unsupported PLY format"):
        load_ply_stl(hdr, parser="gpu")


# ---- vertex-colour raster ----------------------------------------------------------------------------------------
def _rot(n, seed):
    return rotation_matrices(synth.random_view_transforms(n, seed=seed))


def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _rgba(c):
    return _t(np.concatenate([c, np.full((len(c), 1), 255, np.uint8)], 1))


def _render(scans, rot, mode, h=96, w=80):
    return ops.raster_multiscan(scans, _t(rot.reshape(-1, 9)), h, w, mode, want_f32=True, want_tri=True)


@pytest.mark.parametrize("mode", ["RGB+depth", "RGB"])
def test_vertex_colours_match_the_rule_on_the_oracle(lib, face, mode):
    v, _, t, c = face
    rot = _rot(6, 4)
    out = _render([(_t(v), None, _t(t), None, _rgba(c))], rot, mode)
    img, tri, _ = native.raster_multiview(v, None, t, None, rot, 96, 80, mode)
    _same(out["tri"], tri)
    rgb = mesh_ref.shade_vertex_colors(v, t, c, rot, tri, 96, 80)
    u8 = out["u8"].cpu().numpy()
    assert np.array_equal(u8[..., :3], rgb)
    ref = img.copy()
    ref[..., :3] = rgb.astype(np.float32) / np.float32(255)
    _same(out["f32"], ref)
    if mode == "RGB+depth":  # depth channel unchanged
        assert np.array_equal(u8[..., 3], _render([(_t(v), None, _t(t), None)], rot, mode)["u8"].cpu().numpy()[..., 3])


@pytest.mark.parametrize("mode", ["geometry+depth", "depth", "geometry"])
def test_other_modes_ignore_colours(lib, face, mode):
    v, _, t, c = face
    rot = _rot(5, 8)
    a = _render([(_t(v), None, _t(t), None, _rgba(c))], rot, mode)
    b = _render([(_t(v), None, _t(t), None)], rot, mode)
    _same(a["u8"], b["u8"])
    _same(a["f32"], b["f32"])


def test_constant_colour_and_texture_wins(lib, face):
    v, uv, t, c = face
    rot = _rot(4, 2)
    const = np.tile(np.array([[17, 140, 231]], np.uint8), (len(v), 1))
    out = _render([(_t(v), None, _t(t), None, _rgba(const))], rot, "RGB")
    u8, tri = out["u8"].cpu().numpy(), out["tri"].cpu().numpy()
    assert (tri >= 0).sum() > 1000
    assert (u8[tri >= 0][:, :3] == [17, 140, 231]).all() and (u8[tri < 0][:, :3] == 255).all()
    tex = np.concatenate([synth.face_texture(64, seed=1), np.full((64, 64, 1), 255, np.uint8)], 2)
    textured = _render([(_t(v), _t(uv), _t(t), _t(tex))], rot, "RGB+depth")
    both = _render([(_t(v), _t(uv), _t(t), _t(tex), _rgba(c))], rot, "RGB+depth")
    _same(both["u8"], textured["u8"])
    _same(both["f32"], textured["f32"])


def test_multiscan_pass_mixes_obj_ply_stl(lib, tmp_path, face):
    v, uv, t, c = face
    tex = synth.face_texture(128, seed=2)
    obj = load_obj(synth.write_obj(tmp_path / "a.obj", v, uv, t, tex))
    ply = load_mesh(synth.write_ply(tmp_path / "b.ply", v[::-1].copy(), len(v) - 1 - t, c))
    stl = load_mesh(synth.write_stl(tmp_path / "c.stl", v * 0.9, t))
    tex4 = np.concatenate([obj.texture, np.full(obj.texture.shape[:2] + (1,), 255, np.uint8)], 2)
    scans = [(_t(obj.verts), _t(obj.uvs), _t(obj.tris), _t(tex4), None),
             (_t(ply.verts), None, _t(ply.tris), None, _rgba(ply.colors)),
             (_t(stl.verts), None, _t(stl.tris), None)]
    rot = _rot(15, 6)
    for mode in ("RGB+depth", "geometry+depth"):
        both = _render(scans, rot, mode)
        for s, scan in enumerate(scans):
            one = _render([scan], rot[5 * s:5 * s + 5], mode)
            for k in ("u8", "f32", "tri"):
                _same(both[k][5 * s:5 * s + 5], one[k])


# ---- pipeline ----------------------------------------------------------------------------------------------------
def _pipe(name="dtu3d", mode="RGB+depth", n_lm=73, **kw):
    return create_pipeline(name, n_views=8, weights=seeded_state_dict(n_lm, mode, 3), seed=5, n_hypotheses=4,
                           verbose=False, image_size=(128, 128), channel_mode=mode, **kw)


@pytest.fixture(scope="module")
def files(tmp_path_factory, face):
    d = tmp_path_factory.mktemp("scans")
    v, uv, t, c = face
    plain = load_obj(synth.write_obj(d / "plain.obj", v, None, t))  # coordinates as an OBJ file rounds them
    return {"obj": synth.write_obj(d / "a.obj", v, uv, t, synth.face_texture(128, seed=3)),
            "ply": synth.write_ply(d / "b.ply", plain.verts, plain.tris, c),
            "stl": synth.write_stl(d / "c.stl", plain.verts, plain.tris),
            "plain": d / "plain.obj"}


@pytest.mark.parametrize("parser", ["host", "gpu"])
def test_files_equal_predict_mesh_on_the_same_arrays(lib, files, parser):
    dm = _pipe(scan_formats=FORMATS, obj_parser=parser)
    for k in ("ply", "stl"):
        m = load_ply_stl(files[k])
        _same(dm.predict_one_file(files[k]), dm.predict_mesh(m))


@pytest.mark.parametrize("name,mode,n_lm", [("BU3DFE", "geometry+depth", 84), ("BU3DFE", "depth", 84),
                                            ("dtu3d", "depth", 73)])
def test_stl_equals_the_untextured_obj(lib, files, name, mode, n_lm):
    dm = _pipe(name, mode, n_lm, scan_formats=FORMATS)
    _same(dm.predict_one_file(files["stl"]), dm.predict_one_file(files["plain"]))


def test_coloured_ply_teacher_forced(lib, files):
    dm = _pipe(scan_formats=FORMATS)
    tr = synth.random_view_transforms(8, seed=21)
    dm.renderer_3d.transforms = tr
    lm = dm.predict_one_file(files["ply"])
    mesh = load_mesh(files["ply"])
    dmesh = dm.renderer_3d.upload(mesh)
    u8 = dm.renderer_3d.render_device(dmesh, tr)["u8"]
    assert (u8[..., :3] != 255).any(axis=-1).sum() > 1000  # the colours reach the image
    peaks = dm.predictor_2d.predict_landmarks_device(u8).cpu().numpy()
    starts, ends = stages.landmark_lines(128, peaks, tr)
    ref_lm, ref_err, _ = stages.landmarks_from_lines(peaks, starts, ends, dm.estimator_3d.seeded_draws(73))
    ref_snap, _ = native.snap_to_mesh(mesh.verts, mesh.tris, ref_lm)
    assert np.abs(lm - ref_snap).max() <= 1e-6
    assert abs(dm.last_error - ref_err) <= 1e-6 * max(1.0, abs(ref_err))


@pytest.mark.parametrize("parser", ["host", "gpu"])
@pytest.mark.parametrize("pass_pixels", [0, 3 * 8 * 128 * 128])
def test_predict_files_and_folder_mixed_formats(lib, monkeypatch, tmp_path, face, parser, pass_pixels):
    monkeypatch.setattr(gp, "PASS_PIXELS", pass_pixels)
    v, uv, t, c = face
    paths = [synth.write_obj(tmp_path / "a.obj", v, uv, t, synth.face_texture(64, seed=1)),
             synth.write_ply(tmp_path / "b.ply", v * 0.8, t, c, fmt="binary_big_endian"),
             synth.write_stl(tmp_path / "c.STL", v * 0.9, t),
             synth.write_ply(tmp_path / "d.ply", v, t, None, fmt="ascii"),
             synth.write_stl(tmp_path / "e.stl", v * 1.1, t, binary=False)]
    (tmp_path / "notes.txt").write_text("not a scan")
    dm = _pipe(scan_formats=FORMATS, obj_parser=parser)
    assert dm._scans_per_pass() == (1 if pass_pixels == 0 else 3)
    ref = [dm.predict_one_file(p) for p in paths]
    got = dm.predict_files([paths[0], tmp_path / "missing.ply", *paths[1:]])
    for x, y in zip(got, [ref[0], None, *ref[1:]]):
        _same(x, y)
    out = dm.predict_folder(tmp_path, out=tmp_path / "lm")
    assert list(out) == sorted(paths)
    for p in paths:
        _same(out[p], ref[paths.index(p)])
    assert (tmp_path / "lm" / "c_dtu3d.txt").exists()


def test_pre_align_with_a_ply(lib, files):
    cfg = {"align_center_of_mass": True, "rot_x": 10, "rot_y": -20, "rot_z": 5, "scale": 1.1}
    dm = _pipe(scan_formats=FORMATS, pre_align=cfg)
    m = load_ply_stl(files["ply"])
    lm = dm.predict_one_file(files["ply"])
    _same(lm, dm.predict_mesh(m))
    assert not np.array_equal(lm, _pipe(scan_formats=FORMATS).predict_one_file(files["ply"]))


def test_default_pipeline_rejects_ply_and_stl(lib, files):
    dm = _pipe()
    assert dm.scan_formats == ("obj",)
    for k in ("ply", "stl"):
        with pytest.raises(ValueError, match=r"is not an .obj file. Only .obj files are supported."):
            dm.predict_one_file(files[k])
        with pytest.raises(ValueError, match=r"is not an .obj file. Only .obj files are supported."):
            dm.predict_files([files[k]])
    with pytest.raises(ValueError, match="Unknown scan format"):
        _pipe(scan_formats=("obj", "wrl"))
    only_stl = _pipe(scan_formats=("stl",))
    with pytest.raises(ValueError, match="Only .stl files are supported"):
        only_stl.predict_one_file(files["obj"])
    assert only_stl.predict_one_file(files["stl"]).shape == (73, 3)
