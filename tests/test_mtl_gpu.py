"""Texture pages on the GPU (DESIGN.md 7g): paged rasterisation against the C oracle rendered once per page, passes
that mix paged and other scans, and the pipeline's texture_source="mtl" in every entry point."""
import os

import numpy as np
import pytest
import torch

import mtl_ref
from mvlm_b200 import ops, synth
from mvlm_b200.io_mesh import load_mesh
from mvlm_b200.io_obj import Mesh, load_obj
from mvlm_b200.pipeline import create_pipeline
from mvlm_b200.pipeline import general_pipeline as gp
from mvlm_b200.utils.render3d import DeviceMesh, rotation_matrices
from mvlm_b200.weights import seeded_state_dict
from oracle import native

pytestmark = pytest.mark.gpu

DEV = "cuda"
MODES = ["RGB+depth", "geometry+depth", "RGB", "depth", "geometry"]


def _np(a):
    return a.cpu().numpy() if isinstance(a, torch.Tensor) else a


def _same(a, b):
    a, b = _np(a), _np(b)
    assert (a is None) == (b is None)
    if a is not None:
        assert a.dtype == b.dtype and a.shape == b.shape
        assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _t(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _rgba(img):
    return np.concatenate([img, np.full(img.shape[:2] + (1,), 255, np.uint8)], 2)


@pytest.fixture(scope="module")
def paged():
    """Face mesh with uv wrap (coordinates outside [0, 1)), four pages of different sizes and an untextured band."""
    v, uv, t = synth.face_mesh(grid=90, seed=7)
    uv = (uv * 1.7 - 0.35).astype(np.float32)
    tri_page = ((np.arange(len(t)) // 37) % 4).astype(np.int32)
    tri_page[(np.arange(len(t)) // 101) % 5 == 3] = -1
    pages = [synth.face_texture(s, seed=s) for s in (64, 128, 48, 96)]
    pages[2] = pages[2][:, :40].copy()  # not square
    return v, uv, t, pages, tri_page


def _render_paged(v, uv, t, pages, tri_page, rot, mode, h=96, w=80):
    d = DeviceMesh(Mesh(verts=v, tris=t, uvs=uv, texture=None, pages=pages, tri_page=tri_page), torch.device(DEV))
    texels, table = d.paged()
    return ops.raster_multiscan([(d.verts, d.uvs, d.tris, texels, None, table)], _t(rot.reshape(-1, 9)), h, w, mode,
                                want_f32=True, want_tri=True)


@pytest.mark.parametrize("mode", MODES)
def test_paged_images_match_the_oracle_per_page(lib, paged, mode):
    v, uv, t, pages, tri_page = paged
    rot = rotation_matrices(synth.random_view_transforms(6, seed=3))
    out = _render_paged(v, uv, t, pages, tri_page, rot, mode)
    base, tri, _ = native.raster_multiview(v, uv, t, None, rot, 96, 80, mode)
    _same(out["tri"], tri)
    images = [native.raster_multiview(v, uv, t, p, rot, 96, 80, mode)[0] for p in pages]
    ref = mtl_ref.paged_image(images, tri, tri_page, base)
    _same(out["f32"], ref)
    c = ref.shape[-1]
    assert np.array_equal(out["u8"].cpu().numpy()[..., :c], np.rint(ref * 255).astype(np.uint8))
    if mode in ("RGB+depth", "RGB"):  # every page and the white band reach the image
        page = np.where(tri >= 0, tri_page[np.maximum(tri, 0)], -2)
        assert all((page == p).sum() > 100 for p in range(-1, 4))


def test_one_page_equals_the_single_texture_path(lib, paged):
    v, uv, t, pages, _ = paged
    rot = rotation_matrices(synth.random_view_transforms(5, seed=8))
    for mode in ("RGB+depth", "RGB"):
        one = _render_paged(v, uv, t, [pages[1]], np.zeros(len(t), np.int32), rot, mode)
        single = ops.raster_multiscan([(_t(v), _t(uv), _t(t), _t(_rgba(pages[1])))], _t(rot.reshape(-1, 9)), 96, 80, mode,
                                      want_f32=True, want_tri=True)
        for k in ("u8", "f32", "tri"):
            _same(one[k], single[k])


def test_pass_mixes_paged_textured_coloured_and_plain(lib, monkeypatch, tmp_path, paged):
    v, uv, t, pages, tri_page = paged
    col = np.random.RandomState(2).randint(0, 256, (len(v), 3)).astype(np.uint8)
    meshes = [Mesh(verts=v, tris=t, uvs=uv, texture=None, pages=pages, tri_page=tri_page),
              load_obj(synth.write_obj(tmp_path / "a.obj", v * 0.9, uv, t, synth.face_texture(64, seed=4))),
              load_mesh(synth.write_ply(tmp_path / "b.ply", v, t, col)),
              Mesh(verts=v * 1.05, tris=t, uvs=None, texture=None),
              Mesh(verts=v[::-1].copy(), tris=(len(v) - 1 - t).astype(np.int32), uvs=uv[::-1].copy(), texture=None,
                   pages=pages[::-1], tri_page=np.where(tri_page < 0, -1, 3 - tri_page).astype(np.int32))]
    dm = create_pipeline("dtu3d", n_views=8, weights=seeded_state_dict(73, "RGB+depth", 3), seed=5, n_hypotheses=4,
                         verbose=False, image_size=(128, 128), scan_formats=("obj", "ply"))
    r = dm.renderer_3d
    tr = [synth.random_view_transforms(4, seed=s) for s in range(len(meshes))]
    d = [r.upload(m) for m in meshes]
    both = {k: x.clone() for k, x in r.render_pass(d, tr, want_f32=True, want_tri=True).items() if x is not None}
    for s in range(len(meshes)):
        one = r.render_pass([d[s]], [tr[s]], want_f32=True, want_tri=True)
        for k in ("u8", "f32", "tri"):
            _same(both[k][4 * s:4 * s + 4], one[k])
    # the batch driver with several scans per pass gives each scan its own landmarks
    monkeypatch.setattr(gp, "PASS_PIXELS", 5 * 8 * 128 * 128)
    assert dm._scans_per_pass() == 5
    got = dm.predict_meshes(meshes)
    for m, lm in zip(meshes, got):
        _same(lm, dm.predict_mesh(m))


# ---- device parser -----------------------------------------------------------------------------------------------
def _device_equals_host(path, on_device=True):
    g = load_obj(path, parser="gpu", texture_source="mtl")
    h = load_obj(path, parser="host", texture_source="mtl")
    assert isinstance(g.verts, torch.Tensor) == on_device
    if on_device:
        g.geometry_ready.synchronize()
    for a, b in ((g.verts, h.verts), (g.uvs, h.uvs), (g.tris, h.tris), (g.tri_page, h.tri_page), (g.texture, h.texture)):
        _same(a, b)
    assert (g.pages is None) == (h.pages is None)
    for a, b in zip(g.pages or (), h.pages or ()):
        _same(a, b)
    return g, h


@pytest.mark.parametrize("n_mat", [1, 3, 300])
def test_device_parser_materials_equal_host(lib, tmp_path, n_mat):
    v, uv, t = synth.face_mesh(grid=70, seed=n_mat)
    rng = np.random.RandomState(n_mat)
    runs = rng.randint(1, 40, len(t))  # groups of random lengths, some untextured, materials reused
    tri_page = np.repeat(rng.randint(-1, n_mat, len(t)), runs)[:len(t)].astype(np.int32)
    pages = [rng.randint(0, 256, (3 + i % 5, 2 + i % 7, 3)).astype(np.uint8) for i in range(n_mat)]
    p = synth.write_obj_mtl(tmp_path / "s.obj", v, uv, t, pages, tri_page, formats=["png"] * n_mat)
    g, h = _device_equals_host(p)
    assert n_mat == 1 or h.pages is not None
    if n_mat == 3:  # faces before the first usemtl, and a usemtl line without faces
        text = p.read_text()
        first = text.index("usemtl")
        p.write_text(text[:first] + text[text.index("\n", first) + 1:] + "usemtl page2\n")
        g, h = _device_equals_host(p)
        assert (h.tri_page[:5] == -1).all()


def test_device_parser_materials_at_config4_size(lib, tmp_path):
    v, uv, t = synth.face_mesh(grid=1001, seed=3)  # 2M triangles
    tri_page = (np.arange(len(t)) * 4 // len(t)).astype(np.int32)
    tri_page[(np.arange(len(t)) // 1000) % 7 == 3] = -1
    pages = [synth.face_texture(s, seed=s) for s in (16, 24, 32, 8)]
    _device_equals_host(synth.write_obj_mtl(tmp_path / "big.obj", v, uv, t, pages, tri_page, formats=["png"] * 4))


def test_device_parser_material_fallbacks(lib, tmp_path, capsys):
    v, uv, t = synth.face_mesh(grid=20, seed=4)
    pages = [synth.face_texture(8, seed=1), synth.face_texture(16, seed=2)]
    p = synth.write_obj_mtl(tmp_path / "s.obj", v, uv, t, pages, (np.arange(len(t)) % 2).astype(np.int32),
                            formats=["png", "png"])
    text = p.read_text()
    p.write_text(text + "usemtl page0\n" * 70000)  # more name lines than the device parser keeps: host arrays
    _device_equals_host(p, on_device=False)
    p.write_text(text.replace("v ", "v 1.00000000000000000001 0 0\nv ", 1))  # 21 digits: the host parses it
    _device_equals_host(p, on_device=False)
    # no usable page: the device arrays with the <stem>.jpg rule
    (tmp_path / "s.mtl").write_text("newmtl page0\nmap_Kd gone.png\nnewmtl page1\nKd 1 1 1\n")
    p.write_text(text)
    g, h = _device_equals_host(p)
    assert g.texture is None and g.pages is None and "gone.png" in capsys.readouterr().out


# ---- pipeline ----------------------------------------------------------------------------------------------------
def _pipe(**kw):
    return create_pipeline("dtu3d", n_views=8, weights=seeded_state_dict(73, "RGB+depth", 3), seed=5, n_hypotheses=4,
                           verbose=False, image_size=(128, 128), transforms=synth.random_view_transforms(8, seed=13),
                           **kw)


@pytest.fixture(scope="module")
def scans(tmp_path_factory):
    d = tmp_path_factory.mktemp("mtl")
    v, uv, t = synth.face_mesh(grid=120, seed=11)
    grid = np.arange(len(t)) * 4 // len(t)
    # 256^2 and larger: nvJPEG and libjpeg-turbo agree within the decoder test's tolerance (smaller busy pages differ more)
    pages = [synth.face_texture(s, seed=40 + s) for s in (512, 256, 384, 320)]
    out = {"jpg": synth.write_obj_mtl(d / "jpg.obj", v, uv, t, pages, grid),
           "png": synth.write_obj_mtl(d / "png.obj", v * 0.95, uv, t, pages, grid, formats=["png"] * 4)}
    # an MTL that names <stem>.jpg for every face, and the same scan with <stem>.jpg alone
    one = d / "one"
    one.mkdir()
    out["one"] = synth.write_obj_mtl(one / "one.obj", v, uv, t, [pages[0]], np.zeros(len(t), np.int32))
    (one / "one_0.jpg").rename(one / "one.jpg")
    (one / "one.mtl").write_text((one / "one.mtl").read_text().replace("one_0.jpg", "one.jpg"))
    out["plain"] = d / "plain.obj"
    (d / "plain.obj").write_text((one / "one.obj").read_text().replace("mtllib one.mtl\n", ""))
    (d / "plain.jpg").write_bytes((one / "one.jpg").read_bytes())
    return out


def test_stem_and_mtl_agree_on_a_stem_jpg_scan(lib, scans):
    stem, mtl = _pipe(), _pipe(texture_source="mtl")
    assert stem.texture_source == "stem" and mtl.texture_source == "mtl"
    want = stem.predict_one_file(scans["one"])
    _same(mtl.predict_one_file(scans["one"]), want)
    _same(stem.predict_one_file(scans["plain"]), want)
    # with "stem" a scan with only an MTL renders untextured, exactly as before
    untextured = load_obj(scans["jpg"])
    assert untextured.texture is None and untextured.pages is None
    _same(stem.predict_one_file(scans["jpg"]), stem.predict_mesh(untextured))
    assert not np.array_equal(mtl.predict_one_file(scans["jpg"]), stem.predict_one_file(scans["jpg"]))
    with pytest.raises(ValueError, match="Unknown texture source"):
        _pipe(texture_source="jpg")


@pytest.mark.parametrize("parser", ["host", "gpu"])
@pytest.mark.parametrize("pass_pixels", [0, 3 * 8 * 128 * 128])
def test_entry_points_with_mtl(lib, monkeypatch, tmp_path, scans, parser, pass_pixels):
    monkeypatch.setattr(gp, "PASS_PIXELS", pass_pixels)
    dm = _pipe(texture_source="mtl", obj_parser=parser)
    paths = [scans["jpg"], scans["png"], scans["one"], scans["plain"]]
    ref = [dm.predict_mesh(load_obj(p, texture_source="mtl")) for p in paths]
    for p, want in zip(paths, ref):
        _same(dm.predict_one_file(p), want)
    for got, want in zip(dm.predict_files(paths), ref):
        _same(got, want)
    folder = scans["jpg"].parent
    out = dm.predict_folder(folder, out=tmp_path / "lm")
    for p in (scans["jpg"], scans["png"], scans["plain"]):
        _same(out[p], ref[paths.index(p)])
    # the seam renderer reads the pages too
    seams = _pipe(texture_source="mtl", obj_parser=parser, render_image_stack=False)
    img, _, mesh = seams.renderer_3d.multiview_render(scans["jpg"])
    assert mesh.pages is not None and len(mesh.pages) == 4
    dmesh = dm.renderer_3d.upload(load_obj(scans["jpg"], texture_source="mtl"))
    f32 = dm.renderer_3d.render_device(dmesh, seams.renderer_3d.generate_3d_transformations(), want_f32=True)["f32"]
    _same(img, f32)


def test_nvjpeg_pages(lib, scans):
    a = load_obj(scans["jpg"], texture_source="mtl")
    b = load_obj(scans["jpg"], texture_source="mtl", texture_decoder="nvjpeg")
    assert all(isinstance(p, torch.Tensor) and p.is_cuda for p in b.pages) and b.texture_ready is not None
    b.texture_ready.synchronize()
    _same(a.tri_page, b.tri_page)
    for x, y in zip(a.pages, b.pages):
        diff = np.abs(y.cpu().numpy().astype(np.int32) - x.astype(np.int32))
        assert x.shape == tuple(y.shape)
        assert diff.mean() <= 5.0 and (diff > 32).mean() <= 0.02, (diff.max(), diff.mean())
    png = load_obj(scans["png"], texture_source="mtl", texture_decoder="nvjpeg")  # PNG pages go through PIL
    assert all(isinstance(p, np.ndarray) for p in png.pages)
    for parser in ("host", "gpu"):
        dm = _pipe(texture_source="mtl", texture_decoder="nvjpeg", obj_parser=parser)
        one = dm.predict_one_file(scans["jpg"])
        assert np.isfinite(one).all()
        assert all(np.array_equal(one, m) for m in dm.predict_files([scans["jpg"]] * 3))


def test_view_split_upload_carries_pages(lib, scans):
    """World size 1 over NCCL: the sharded upload carries the pages and the page of every triangle, and the view-split
    path equals predict_mesh for a paged scan."""
    import torch.distributed as dist

    from mvlm_b200 import sharding

    dm = _pipe(texture_source="mtl")
    mesh = load_obj(scans["jpg"], texture_source="mtl")
    tr = synth.random_view_transforms(8, seed=13)
    single = dm.predict_mesh(mesh)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29541")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        r = dm.renderer_3d
        sharded = sharding.upload_mesh_sharded(r, mesh)
        _same(r.render_device(sharded, tr)["u8"].clone(), r.render_device(r.upload(mesh), tr)["u8"])
        split = sharding.predict_mesh_view_split(dm, mesh, tr)
    finally:
        if created:
            dist.destroy_process_group()
    _same(split, single)
