"""PLY / STL scan loader on the host (csrc/mesh_loader.cu) against the numpy restatement tests/mesh_ref.py, the weld
rules on hand-written soups, and every error message.  No GPU."""
import struct

import numpy as np
import pytest

import mesh_ref
from mvlm_b200 import synth
from mvlm_b200.io_mesh import check_scan_file, check_scan_path, is_scan_file, load_mesh, load_ply_stl


def _same(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def _check_ply(path):
    m = load_ply_stl(path)
    v, c, t = mesh_ref.read_ply(path)
    _same(m.verts, v)
    _same(m.tris, t)
    if c is None:
        assert m.colors is None
    else:
        _same(m.colors, c)
    return m


def _check_stl(path):
    m = load_ply_stl(path)
    v, t = mesh_ref.read_stl(path)
    _same(m.verts, v)
    _same(m.tris, t)
    assert m.colors is None and m.uvs is None
    return m


@pytest.fixture(scope="module")
def face():
    v, _, t = synth.face_mesh(grid=24, seed=7)
    rng = np.random.RandomState(3)
    return v, t, rng.randint(0, 256, (len(v), 3)).astype(np.uint8)


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
@pytest.mark.parametrize("pos_type", ["float", "double"])
@pytest.mark.parametrize("with_colors", [False, True])
def test_ply_matches_reference(lib, tmp_path, face, fmt, pos_type, with_colors):
    v, t, c = face
    p = synth.write_ply(tmp_path / "s.ply", v, t, c if with_colors else None, fmt=fmt, pos_type=pos_type)
    m = _check_ply(p)
    assert m.verts.shape == v.shape and np.array_equal(m.tris, t)
    if pos_type == "float":
        _same(m.verts, v)


@pytest.mark.parametrize("fmt", ["ascii", "binary_little_endian", "binary_big_endian"])
@pytest.mark.parametrize("count_type,index_type", [("uchar", "int"), ("int", "uint"), ("uint", "int"),
                                                   ("uint8", "int32"), ("ushort", "ushort")])
def test_ply_polygons_and_index_types(lib, tmp_path, face, fmt, count_type, index_type):
    v, t, _ = face
    # quads, pentagons, a 2-corner and a 0-corner face (no triangle), and triangles
    faces = [list(t[0]) + [5], [1, 2, 3, 4, 6], [7, 8], [], list(t[1])] + [list(x) for x in t[2:40]]
    p = synth.write_ply(tmp_path / "poly.ply", v, faces, fmt=fmt, count_type=count_type, index_type=index_type)
    m = _check_ply(p)
    assert len(m.tris) == 2 + 3 + 1 + 38
    assert m.tris[:2].tolist() == [[t[0][0], t[0][1], t[0][2]], [t[0][0], t[0][2], 5]]  # fan (0, k, k + 1)


@pytest.mark.parametrize("crlf", [False, True])
def test_ply_skips_other_properties_and_elements(lib, tmp_path, crlf):
    nl = "\r\n" if crlf else "\n"
    text = nl.join([
        "ply", "format ascii 1.0", "comment scanner export", "obj_info some info",
        "element material 1", "property uchar ambient_red", "property list uchar float params",
        "element vertex 4", "property float nx", "property double x", "property float y", "property int16 z",
        "property uchar red", "property uchar green", "property uchar blue", "property uchar alpha",
        "property float confidence",
        "element face 2", "property uchar flags", "property list uchar int vertex_index",
        "property list uchar float texcoord",
        "element edge 1", "property list int int vertex_pair",
        "end_header",
        "7 2 0.5 1.5",
        "0 0.1 0.2 3 10 20 30 255 0.9", "0 1.25 0.5 -4 40 50 60 255 0.9",
        "1 2.5 7.75 5 70 80 90 128 0.1", "1 -1e-3 3 0 100 110 120 0 0.5",
        "1 3 0 1 2 6 0 0 1 0 1 1", "0 4 0 2 3 1 0",
        "2 0 3", ""])
    (tmp_path / "x.ply").write_bytes(text.encode())
    m = _check_ply(tmp_path / "x.ply")
    assert m.tris.tolist() == [[0, 1, 2], [0, 2, 3], [0, 3, 1]]
    assert m.colors.tolist() == [[10, 20, 30], [40, 50, 60], [70, 80, 90], [100, 110, 120]]
    assert m.verts[1].tolist() == [1.25, 0.5, -4.0]


def test_ply_colors_only_when_all_uchar(lib, tmp_path, face):
    v, t, c = face
    p = synth.write_ply(tmp_path / "c.ply", v, t, c, fmt="ascii")
    p.write_bytes(p.read_bytes().replace(b"property uchar blue", b"property ushort blue"))
    m = _check_ply(p)
    assert m.colors is None


def test_stl_binary_and_ascii_match_reference(lib, tmp_path, face):
    v, t, _ = face
    a = _check_stl(synth.write_stl(tmp_path / "b.stl", v, t))
    b = _check_stl(synth.write_stl(tmp_path / "a.stl", v, t, binary=False))
    _same(a.verts, b.verts)
    _same(a.tris, b.tris)
    # the weld restores the indexed mesh up to the order of first occurrence; triangles keep their order
    _same(a.verts[a.tris], v[t])
    # a binary STL whose header starts with "solid" is still binary (the size rule decides)
    c = _check_stl(synth.write_stl(tmp_path / "s.stl", v, t, header=b"solid exported by a scanner"))
    _same(c.verts, a.verts)


def test_stl_ascii_crlf_and_several_solids(lib, tmp_path):
    facet = "facet normal 0 0 1\r\n outer loop\r\n  vertex {} \r\n  vertex {}\r\n  vertex {}\r\n endloop\r\nendfacet\r\n"
    text = ("solid first part\r\n" + facet.format("0 0 0", "1 0 0", "0 1 0") + "endsolid first part\r\n"
            + "solid second\r\n" + facet.format("1 0 0", "+1 1 0", "0 1 0") + "\r\n" + "endsolid\r\n")
    (tmp_path / "x.stl").write_bytes(text.encode())
    m = _check_stl(tmp_path / "x.stl")
    assert m.verts.tolist() == [[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0]]
    assert m.tris.tolist() == [[0, 1, 2], [1, 3, 2]]


def _binary_stl(path, corners, header=b"x"):
    c = np.asarray(corners, np.float32).reshape(-1, 9)
    rec = np.zeros(len(c), dtype=[("n", "<f4", (3,)), ("v", "<f4", (9,)), ("a", "<u2")])
    rec["v"] = c
    rec["a"] = 0xBEEF  # the attribute word is ignored
    path.write_bytes(header.ljust(80, b"\0") + struct.pack("<I", len(c)) + rec.tobytes())
    return path


def test_weld_first_occurrence_on_a_hand_written_soup(lib, tmp_path):
    A, B, C, D, E = [5, 0, 0], [0, 5, 0], [0, 0, 5], [1, 1, 1], [2, 2, 2]
    p = _binary_stl(tmp_path / "w.stl", [C, A, B, B, D, A, E, C, D])
    m = _check_stl(p)
    assert m.verts.tolist() == [C, A, B, D, E]  # order of first occurrence in corner order
    assert m.tris.tolist() == [[0, 1, 2], [2, 3, 1], [4, 0, 3]]


def test_weld_signed_zero_nan_duplicates_degenerate(lib, tmp_path):
    nan = float("nan")
    soup = [[-0.0, 0, 0], [1, 0, 0], [0, 1, 0],      # -0.0 first: the vertex keeps -0.0
            [0.0, 0, 0], [1, 0, 0], [0, 1, 0],       # duplicate facet (with +0.0): kept, same ids
            [nan, 0, 0], [1, 0, 0], [nan, 0, 0],     # NaN corners never merge: two vertices, facet kept
            [1, 0, 0], [0, 1, 0], [1, 0, 0],         # degenerate after the weld: dropped
            [2, 2, 2], [2, 2, 2], [2, 2, 2],         # fully collapsed: dropped, its vertex stays
            [0, 1, 0], [1, 0, 0], [0, -0.0, 0.0]]    # (0,-0,0) == (0,0,0)
    m = _check_stl(_binary_stl(tmp_path / "z.stl", soup))
    assert len(m.verts) == 6
    assert np.signbit(m.verts[0, 0]) and np.isnan(m.verts[3, 0]) and np.isnan(m.verts[4, 0])
    assert m.tris.tolist() == [[0, 1, 2], [0, 1, 2], [3, 1, 4], [2, 1, 0]]


@pytest.mark.parametrize("suffix", [".ply", ".stl"])
def test_missing_file(lib, tmp_path, suffix):
    with pytest.raises(ValueError, match="does not exist"):
        load_ply_stl(tmp_path / ("nope" + suffix))


def _err(lib, path):
    import ctypes as C

    h = C.c_void_p()
    assert lib.mvlm_mesh_load(str(path).encode(), 0, C.byref(h)) != 0
    with pytest.raises(ValueError) as e:
        load_ply_stl(path)
    assert str(e.value) == lib.mvlm_last_error().decode()
    return str(e.value)


def _ply(tmp_path, header, body, name="e.ply"):
    p = tmp_path / name
    p.write_bytes(("\n".join(header) + "\nend_header\n").encode() + body)
    return p


def test_error_messages(lib, tmp_path):
    vtx = ["element vertex 3", "property float x", "property float y", "property float z"]
    fce = ["element face 1", "property list uchar int vertex_indices"]
    asc = b"0 0 0\n1 0 0\n0 1 0\n"
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + ["element face 0", fce[1]], asc)
    assert _err(lib, p) == f"File {p} does not contain any points."
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + fce, asc + b"3 0 1 3\n")
    assert _err(lib, p) == f"mvlm_mesh_load: face references vertex 3 of 3 in {p}"
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + fce, asc + b"3 0 -1 2\n")
    assert _err(lib, p) == f"mvlm_mesh_load: face references vertex -1 of 3 in {p}"
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + fce, b"0 0 0\n1 0x 0\n0 1 0\n3 0 1 2\n")
    assert _err(lib, p) == f"mvlm_mesh_load: malformed ASCII number in {p}"
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + fce, asc + b"3 0 1.5 2\n")
    assert "malformed ASCII number" in _err(lib, p)
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + fce, asc + b"3 0 1\n")
    assert "truncated PLY body" in _err(lib, p)
    p = _ply(tmp_path, ["ply", "format binary_little_endian 1.0"] + vtx + fce, b"\0" * 36 + b"\3" + b"\0" * 11)
    assert _err(lib, p) == f"mvlm_mesh_load: truncated binary PLY body in {p}"
    p = _ply(tmp_path, ["ply", "format binary_middle_endian 1.0"] + vtx + fce, b"")
    assert _err(lib, p) == f"mvlm_mesh_load: unsupported PLY format 'binary_middle_endian' in {p}"
    p = _ply(tmp_path, ["ply", "format ascii 1.0", "element vertex 3", "property float128 x"], b"")
    assert _err(lib, p) == f"mvlm_mesh_load: unsupported PLY property type 'float128' in {p}"
    p = _ply(tmp_path, ["ply", "format ascii 1.0", "element vertex 1", "property float x", "property float y"], b"0 0\n")
    assert _err(lib, p) == f"mvlm_mesh_load: malformed PLY header in {p} (vertex element without x y z)"
    p = _ply(tmp_path, ["ply", "format ascii 1.0"] + vtx + ["element face 1", "property list uchar int corners"], asc)
    assert "face element without vertex_indices" in _err(lib, p)
    p = tmp_path / "h.ply"
    p.write_bytes(b"ply\nformat ascii 1.0\nelement vertex 3\n")
    assert _err(lib, p) == f"mvlm_mesh_load: malformed PLY header in {p} (no end_header)"
    p = tmp_path / "n.ply"
    p.write_bytes(b"solid\n")
    assert "is not a PLY file" in _err(lib, p)
    p = tmp_path / "e.stl"
    p.write_bytes(b"solid empty\nendsolid empty\n")
    assert _err(lib, p) == f"File {p} does not contain any points."
    p = tmp_path / "d.stl"
    _binary_stl(p, [[1, 1, 1]] * 3)  # one facet, degenerate after the weld
    assert _err(lib, p) == f"File {p} does not contain any points."
    p = tmp_path / "t.stl"
    p.write_bytes(_binary_stl(tmp_path / "u.stl", [[0, 0, 0], [1, 0, 0], [0, 1, 0]]).read_bytes()[:-1])  # truncated
    assert "is neither a binary STL" in _err(lib, p)
    p = tmp_path / "m.stl"
    p.write_bytes(b"solid x\nfacet normal 0 0 1\nouter loop\nvertex 0 0 0\nvertex 1 0 0\nendloop\nendfacet\nendsolid\n")
    assert "facet without 3 vertices" in _err(lib, p)
    p = tmp_path / "f.stl"
    p.write_bytes(b"solid x\nfacet normal 0 0 1\nouter loop\nvertex 0 0 zero\n")
    assert _err(lib, p) == f"mvlm_mesh_load: malformed ASCII number in {p}"
    p = tmp_path / "x.off"
    p.write_bytes(b"OFF\n")
    assert "is not a .ply or .stl file" in _err(lib, p)


def test_load_mesh_dispatch_and_scan_file_checks(lib, tmp_path, face):
    from pathlib import Path

    v, t, _ = face
    obj = synth.write_obj(tmp_path / "a.obj", v, None, t)
    m = load_mesh(obj)
    assert m.colors is None and m.verts.shape == v.shape
    s = load_mesh(synth.write_stl(tmp_path / "A.STL", v, t))
    assert s.tris.shape == t.shape
    with pytest.raises(ValueError, match="is not an .obj, .ply or .stl file"):
        load_mesh(tmp_path / "a.wrl")
    assert is_scan_file(Path("a.obj"), ("obj",)) and not is_scan_file(Path("a.OBJ"), ("obj",))
    assert not is_scan_file(Path("a.ply"), ("obj",)) and is_scan_file(Path("a.PLY"), ("obj", "ply"))
    assert not is_scan_file(Path("a.stl"), ("obj", "ply"))
    with pytest.raises(ValueError, match=r"^File a.ply is not an .obj file. Only .obj files are supported.$"):
        check_scan_file(Path("a.ply"), ("obj",))
    with pytest.raises(ValueError, match="Only .obj, .ply, .stl files are supported"):
        check_scan_file(Path("a.wrl"), ("obj", "ply", "stl"))
    check_scan_path(tmp_path / "A.STL", ("obj", "stl"))
    with pytest.raises(ValueError, match=r"^File .*A.STL is not an .obj file. Only .obj files are supported.$"):
        check_scan_path(tmp_path / "A.STL", ("obj",))
    with pytest.raises(FileNotFoundError, match=r"^File .* is not a file$"):
        check_scan_path(tmp_path, ("obj",))  # checked before the suffix


def test_mesh_symbols_and_info_layout(lib):
    import ctypes as C

    from mvlm_b200 import _lib

    for name in ("mvlm_mesh_load", "mvlm_mesh_counts", "mvlm_mesh_copy", "mvlm_mesh_free", "mvlm_mesh_parse_device",
                 "mvlm_mesh_parse_write", "mvlm_mesh_parse_workspace_bytes", "mvlm_raster_multiscan_colored"):
        assert hasattr(lib, name)
    assert C.sizeof(_lib.MeshParseInfo) == 32
    # the device decoder's capacity: one scan of 16.7M corners, so about 5.5M facets; non-binary-STL sizes take the host
    assert lib.mvlm_mesh_parse_workspace_bytes(84 + 50 * 5_500_000, 1) > 0
    assert lib.mvlm_mesh_parse_workspace_bytes(84 + 50 * 5_600_000, 1) == 0
    assert lib.mvlm_mesh_parse_workspace_bytes(85, 1) == 0
    assert lib.mvlm_mesh_parse_workspace_bytes(84, 1) == 0
    assert lib.mvlm_mesh_parse_workspace_bytes(1000, 0) >= 1000
