"""OBJ materials on the host (DESIGN.md 7g): mvlm_obj_load_ex's MVLM_OBJ_MATERIALS output against the numpy
restatement (tests/mtl_ref.py), the MTL rules of io_obj and the texture_source option of the loaders."""
import ctypes as C

import numpy as np
import pytest

import mtl_ref
from mvlm_b200 import _lib, synth
from mvlm_b200.io_mesh import load_mesh
from mvlm_b200.io_obj import load_obj, parse_mtl


def _load_ex(lib, path, n_threads, flags=_lib.OBJ_MATERIALS):
    h = C.c_void_p()
    assert lib.mvlm_obj_load_ex(str(path).encode(), n_threads, flags, C.byref(h)) == 0, lib.mvlm_last_error()
    try:
        nv, nt, has_uv = C.c_int(), C.c_int(), C.c_int()
        _lib.check(lib.mvlm_obj_counts(h, C.byref(nv), C.byref(nt), C.byref(has_uv)))
        verts = np.empty((nv.value, 3), np.float32)
        tris = np.empty((nt.value, 3), np.int32)
        uvs = np.empty((nv.value, 2), np.float32) if has_uv.value else None
        _lib.check(lib.mvlm_obj_copy(h, verts.ctypes.data, None if uvs is None else uvs.ctypes.data, tris.ctypes.data))
        if not flags:
            return verts, uvs, tris, None
        tm = np.empty((nt.value,), np.int32)
        n_mat, n_lib = C.c_int(), C.c_int()
        _lib.check(lib.mvlm_obj_materials(h, tm.ctypes.data, C.byref(n_mat), C.byref(n_lib)))
        names = [lib.mvlm_obj_material_name(h, i).decode("utf-8", "surrogateescape") for i in range(n_mat.value)]
        libs = [lib.mvlm_obj_library_name(h, i).decode("utf-8", "surrogateescape") for i in range(n_lib.value)]
        assert lib.mvlm_obj_material_name(h, n_mat.value) is None and lib.mvlm_obj_library_name(h, -1) is None
        return verts, uvs, tris, (tm, names, libs)
    finally:
        lib.mvlm_obj_free(h)


def _check(lib, path, threads=(1, 3, 16)):
    ref = mtl_ref.obj_materials(path)
    base = _load_ex(lib, path, 1, 0)
    for n in threads:
        v, uv, t, (tm, names, libs) = _load_ex(lib, path, n)
        assert np.array_equal(tm, ref[0]) and names == ref[1] and libs == ref[2], n
        for a, b in zip((v, uv, t), base[:3]):  # the flag changes none of mvlm_obj_load's arrays
            assert (a is None and b is None) or np.array_equal(a, b)
    return ref


QUAD = "v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvt 0 0\nvt 1 0\nvt 1 1\nvt 0 1\n"

CASES = {
    "before_between_repeated": QUAD + "f 1/1 2/2 3/3\nusemtl a\nf 1/1 2/2 3/3 4/4\nusemtl b\nf 1/1 3/3 4/4\n"
                                      "usemtl a\nf 2/2 3/3 4/4\nusemtl a\nf 1/1 2/2 4/4\n",
    "usemtl_before_any_face": "mtllib lib one.mtl\nusemtl first\nusemtl second\n" + QUAD + "f 1/1 2/2 3/3\n",
    "unknown_and_spaces": QUAD + "usemtl  my material  \t\nf 1/1 2/2 3/3\nusemtl\tnot defined\nf 1 2 3\n"
                                 "usemtl \nf 1 3 4\nusemtlx c\nf 2 3 4\n",
    "crlf": "mtllib m.mtl\r\n" + QUAD.replace("\n", "\r\n") + "usemtl a\r\nf 1/1 2/2 3/3\r\nusemtl b \r\nf 1 3 4\r\n",
    "o_g_s_interleaved": "mtllib x.mtl\nmtllib sub\\y.mtl\n" + QUAD + "o obj\ng grp\nusemtl a\ns 1\nf 1/1 2/2 3/3\n"
                         "g other\ns off\nf 1/1 3/3 4/4\no two\nusemtl b\ng g3\nf 2/2 3/3 4/4\n",
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_materials_match_the_restatement(lib, tmp_path, case):
    p = tmp_path / "s.obj"
    p.write_bytes(CASES[case].encode())
    _check(lib, p, threads=(1,))


def test_case_values(lib, tmp_path):
    p = tmp_path / "s.obj"
    p.write_bytes(CASES["before_between_repeated"].encode())
    tm, names, libs = _load_ex(lib, p, 1)[3]
    assert tm.tolist() == [-1, 0, 0, 1, 0, 0] and names == ["a", "b"] and libs == []
    p.write_bytes(CASES["unknown_and_spaces"].encode())
    tm, names, _ = _load_ex(lib, p, 1)[3]
    assert names == ["my material", "not defined", ""] and tm.tolist() == [0, 1, 2, 2]
    p.write_bytes(CASES["o_g_s_interleaved"].encode())
    assert _load_ex(lib, p, 1)[3][2] == ["x.mtl", "sub\\y.mtl"]


def _chunk_first_lines(lib, data: bytes, n: int):
    """First line of every chunk after the first, at the offsets mvlm_obj_load itself splits the file."""
    starts = np.zeros(max(n, 16), np.int64)
    k = lib.mvlm_debug_obj_chunk_starts(data, len(data), n, starts.ctypes.data)
    assert k == n
    return [data[s:data.find(b"\n", s)] for s in starts[1:k]]


def test_usemtl_on_chunk_boundaries(lib, tmp_path):
    v, uv, t = synth.face_mesh(grid=60, seed=2)
    rng = np.random.RandomState(4)
    lines = ["mtllib a.mtl"] + [f"v {x:.5f} {y:.5f} {z:.5f}" for x, y, z in v] + [f"vt {a:.5f} {b:.5f}" for a, b in uv]
    for i, (a, b, c) in enumerate(t + 1):
        if i % 2 == 0 and rng.rand() < 0.7:
            lines.append(f"usemtl m{rng.randint(0, 7)}")
        lines.append(f"f {a}/{a} {b}/{b} {c}/{c}")
    data = ("\n".join(lines) + "\n").encode()
    assert len(data) > 1 << 16  # chunked parse
    starts = _chunk_first_lines(lib, data, 16)
    assert any(s.startswith(b"usemtl") for s in starts) and any(s.startswith(b"f ") for s in starts)
    p = tmp_path / "big.obj"
    p.write_bytes(data)
    tm, names, _ = _check(lib, p)
    assert len(names) == 7 and (tm >= 0).sum() > len(tm) // 2


def test_flags_and_symbols(lib, tmp_path):
    for name in ("mvlm_obj_load_ex", "mvlm_obj_materials", "mvlm_obj_material_name", "mvlm_obj_library_name",
                 "mvlm_raster_multiscan_paged"):
        assert hasattr(lib, name)
    assert C.sizeof(_lib.RasterScan) == 64  # the public scan struct is unchanged
    p = tmp_path / "s.obj"
    p.write_bytes(CASES["crlf"].encode())
    h = C.c_void_p()
    assert lib.mvlm_obj_load_ex(str(p).encode(), 1, 2, C.byref(h)) != 0
    assert b"unknown flags" in lib.mvlm_last_error()
    assert lib.mvlm_obj_load(str(p).encode(), 1, C.byref(h)) == 0
    n1, n2 = C.c_int(), C.c_int()
    assert lib.mvlm_obj_materials(h, None, C.byref(n1), C.byref(n2)) != 0
    assert b"without MVLM_OBJ_MATERIALS" in lib.mvlm_last_error()
    lib.mvlm_obj_free(h)
    with pytest.raises(ValueError, match="Unknown texture source"):
        load_obj(p, texture_source="vtk")
    with pytest.raises(ValueError, match="Unknown texture source"):
        load_mesh(p, texture_source="MTL")


# ---- MTL rules ---------------------------------------------------------------------------------------------------
def _img(tmp, name, color, size=(4, 6), fmt=None):
    from PIL import Image

    path = tmp / name
    path.parent.mkdir(parents=True, exist_ok=True)
    Image.fromarray(np.full(size + (3,), color, np.uint8)).save(path, format=fmt)
    return path


def test_parse_mtl(tmp_path):
    (tmp_path / "sub").mkdir()
    mtl = tmp_path / "sub" / "m.mtl"
    mtl.write_bytes(b"# comment\r\nnewmtl  skin tone \r\n\tKd 0.5 0.5 0.5\r\n\tmap_Kd -s 1 1 1 -o 0 0 tex\\a.png\r\n"
                    b"newmtl plain\nKd 1 0 0\nmap_Bump b.png\nd 0.5\n"
                    b"newmtl skin tone\nmap_Kd other.png\n"
                    b"newmtl last\nmap_Kd  c.jpg  \n")
    mats = {"preset": None}
    parse_mtl(mtl, mats)
    assert mats == {"preset": None, "skin tone": tmp_path / "sub" / "tex" / "a.png", "plain": None,
                    "last": tmp_path / "sub" / "c.jpg"}
    with pytest.raises(OSError):
        parse_mtl(tmp_path / "missing.mtl", {})


def _quads(tmp_path, body, mtl):
    (tmp_path / "m.mtl").write_text(mtl)
    p = tmp_path / "s.obj"
    p.write_text("mtllib m.mtl\n" + QUAD + body)
    return p


def test_pages_in_order_of_first_use(tmp_path, capsys):
    _img(tmp_path, "a.png", (10, 20, 30), (4, 6))
    _img(tmp_path, "b.bmp", (40, 50, 60), (3, 5))
    _img(tmp_path, "tex/c.jpg", (200, 100, 0), (8, 8))
    (tmp_path / "bad.png").write_bytes(b"not an image")
    mtl = ("newmtl A\nmap_Kd a.png\nnewmtl B\nmap_Kd b.bmp\nnewmtl A2\nmap_Kd ./a.png\nnewmtl C\nmap_Kd tex\\c.jpg\n"
           "newmtl M\nmap_Kd missing.png\nnewmtl U\nmap_Kd bad.png\nnewmtl K\nKd 1 0 0\n")
    body = ("f 1/1 2/2 3/3\nusemtl B\nf 1/1 2/2 3/3\nusemtl M\nf 1/1 2/2 3/3\nusemtl A\nf 1/1 2/2 3/3 4/4\n"
            "usemtl K\nf 1/1 2/2 3/3\nusemtl A2\nf 1/1 2/2 3/3\nusemtl nope\nf 1/1 2/2 3/3\nusemtl C\nf 1/1 2/2 3/3\n"
            "usemtl U\nf 1/1 2/2 3/3\nusemtl M\nf 1/1 2/2 3/3\n")
    m = load_obj(_quads(tmp_path, body, mtl), texture_source="mtl")
    assert m.texture is None and len(m.pages) == 3
    assert m.tri_page.dtype == np.int32 and m.tri_page.tolist() == [-1, 0, -1, 1, 1, -1, 1, -1, 2, -1, -1]
    assert [p.shape for p in m.pages] == [(3, 5, 3), (4, 6, 3), (8, 8, 3)]
    assert (m.pages[0] == (40, 50, 60)).all() and (m.pages[1] == (10, 20, 30)).all()
    out = capsys.readouterr().out
    assert out.count("missing.png") == 1 and out.count("bad.png") == 1  # reported once per file
    # the default rule ignores the materials: no <stem>.jpg, no texture
    d = load_obj(tmp_path / "s.obj")
    assert d.texture is None and d.pages is None and d.tri_page is None


def test_one_page_is_a_single_texture_scan(tmp_path):
    _img(tmp_path, "s.jpg", (90, 80, 70), (16, 16), "JPEG")
    p = _quads(tmp_path, "usemtl A\nf 1/1 2/2 3/3 4/4\nusemtl B\nf 1/1 3/3 4/4\n",
               "newmtl A\nmap_Kd s.jpg\nnewmtl B\nmap_Kd ./s.jpg\n")
    a, b = load_obj(p, texture_source="mtl"), load_obj(p)
    assert a.pages is None and a.tri_page is None
    assert np.array_equal(a.texture, b.texture)
    for x, y in ((a.verts, b.verts), (a.uvs, b.uvs), (a.tris, b.tris)):
        assert np.array_equal(x, y)
    # one page that some triangles do not use is a paged scan
    p.write_text("mtllib m.mtl\n" + QUAD + "usemtl A\nf 1/1 2/2 3/3\nusemtl K\nf 1/1 3/3 4/4\n")
    c = load_obj(p, texture_source="mtl")
    assert c.texture is None and c.tri_page.tolist() == [0, -1] and len(c.pages) == 1


def test_fallback_to_the_stem_rule(tmp_path, capsys):
    stem = _img(tmp_path, "s.jpg", (1, 2, 3), (5, 5), "JPEG")
    ref = load_obj(_quads(tmp_path, "f 1/1 2/2 3/3\n", "")).texture
    assert ref is not None
    cases = {
        "no_mtllib": (QUAD + "usemtl A\nf 1/1 2/2 3/3\n", None),
        "missing_library": ("mtllib gone.mtl\n" + QUAD + "usemtl A\nf 1/1 2/2 3/3\n", None),
        "no_map_kd": ("mtllib m.mtl\n" + QUAD + "usemtl K\nf 1/1 2/2 3/3\n", "newmtl K\nKd 1 1 1\n"),
        "unreadable_only": ("mtllib m.mtl\n" + QUAD + "usemtl U\nf 1/1 2/2 3/3\n", "newmtl U\nmap_Kd nothing.png\n"),
        "no_usemtl": ("mtllib m.mtl\n" + QUAD + "f 1/1 2/2 3/3\n", "newmtl A\nmap_Kd a.png\n"),
    }
    _img(tmp_path, "a.png", (9, 9, 9))
    for name, (obj, mtl) in cases.items():
        if mtl is not None:
            (tmp_path / "m.mtl").write_text(mtl)
        (tmp_path / "s.obj").write_text(obj)
        m = load_obj(tmp_path / "s.obj", texture_source="mtl")
        assert m.pages is None and np.array_equal(m.texture, ref), name
    assert "gone.mtl" in capsys.readouterr().out
    # the flame rule applies as well
    flame = tmp_path / "flame_x.obj"
    flame.write_text(QUAD + "f 1/1 2/2 3/3\n")
    stem.rename(tmp_path / "mean_texture.jpg")
    assert np.array_equal(load_obj(flame, texture_source="mtl").texture, ref)
    # without texture coordinates there is nothing to texture
    (tmp_path / "m.mtl").write_text("newmtl A\nmap_Kd a.png\n")
    (tmp_path / "s.obj").write_text("mtllib m.mtl\nv 0 0 0\nv 1 0 0\nv 0 1 0\nusemtl A\nf 1 2 3\n")
    m = load_obj(tmp_path / "s.obj", texture_source="mtl")
    assert m.texture is None and m.pages is None


def test_write_obj_mtl_round_trip(lib, tmp_path):
    v, uv, t = synth.face_mesh(grid=20, seed=3)
    tri_page = (np.arange(len(t)) * 4 // len(t)).astype(np.int32)
    tri_page[5:9] = -1
    pages = [synth.face_texture(s, seed=s) for s in (16, 32, 24, 8)]
    p = synth.write_obj_mtl(tmp_path / "f.obj", v, uv, t, pages, tri_page, formats=["jpg", "png", "png", "jpg"])
    m = load_obj(p, texture_source="mtl")
    plain = load_obj(p)
    assert np.array_equal(m.tri_page, tri_page) and np.array_equal(m.tris, plain.tris)
    assert [x.shape for x in m.pages] == [x.shape for x in pages]
    assert np.array_equal(m.pages[1], pages[1]) and np.array_equal(m.pages[2], pages[2])  # PNG is lossless
    from PIL import Image

    assert np.array_equal(m.pages[0], np.asarray(Image.open(tmp_path / "f_0.jpg").convert("RGB")))
