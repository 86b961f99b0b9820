"""The text split the host loaders share (csrc/host_text.cuh line_cuts): the offsets mvlm_obj_load splits at against a
restatement of the rule, and PLY / STL ASCII bodies that load to the same arrays with any thread count.  No GPU."""
import numpy as np
import pytest

import mesh_ref
from mvlm_b200 import synth
from mvlm_b200.io_mesh import load_ply_stl


def _cuts(text: bytes, n: int) -> list:
    """One chunk below 65 536 bytes; else cut i is one past the first '\\n' at or after max(size * i // n, cut i-1),
    or the end of the text when there is none."""
    size = len(text)
    if size < 1 << 16:
        return [0]
    cuts = [0]
    for i in range(1, n):
        nl = text.find(b"\n", max(size * i // n, cuts[-1]))
        cuts.append(size if nl < 0 else nl + 1)
    return cuts


def _short_lines(size: int) -> bytes:
    line = b"v 0.125 -3.5 17\n"
    return (line * (size // len(line) + 1))[:size]


def _texts() -> dict:
    rng = np.random.RandomState(5)
    long_lines = b"\n".join(b"f" * int(k) for k in rng.randint(1, 40000, 12))
    texts = {f"short_{n}": _short_lines(n) for n in (65535, 65536, 65537, 200000)}
    texts["short_no_final_newline"] = _short_lines(100000).rstrip(b"\n") + b"x"
    texts["aligned"] = (b"x" * 15 + b"\n") * (1 << 13)  # size * i // n is a line start for n = 1, 2, 16
    texts["long_lines"] = long_lines + b"\n"
    texts["long_lines_no_final_newline"] = long_lines
    texts["one_line"] = b"y" * 100000
    return texts


@pytest.mark.parametrize("name", sorted(_texts()))
def test_chunk_starts_follow_the_rule(lib, name):
    text = _texts()[name]
    for n in (1, 2, 3, 7, 16):
        starts = np.zeros(16, np.int64)
        k = lib.mvlm_debug_obj_chunk_starts(text, len(text), n, starts.ctypes.data)
        assert starts[:k].tolist() == _cuts(text, n), (name, n)


def _same(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape
    assert np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8))


def test_ascii_ply_and_stl_do_not_depend_on_the_thread_count(lib, tmp_path):
    v, _, t = synth.face_mesh(grid=64, seed=9)
    c = np.random.RandomState(6).randint(0, 256, (len(v), 3)).astype(np.uint8)
    files = [synth.write_ply(tmp_path / "plain.ply", v, t, fmt="ascii"),
             synth.write_ply(tmp_path / "colored.ply", v, t, c, fmt="ascii"),
             synth.write_stl(tmp_path / "s.stl", v, t, binary=False)]
    for p in files:
        data = p.read_bytes()
        body = len(data) - data.index(b"end_header\n") - 11 if p.suffix == ".ply" else len(data)
        assert body > 1 << 16, p  # split into chunks
        if p.suffix == ".ply":
            ref_v, ref_c, ref_t = mesh_ref.read_ply(p)
        else:
            (ref_v, ref_t), ref_c = mesh_ref.read_stl(p), None
        for n in (1, 2, 3, 16):
            m = load_ply_stl(p, n_threads=n)
            _same(m.verts, ref_v)
            _same(m.tris, ref_t)
            if ref_c is None:
                assert m.colors is None
            else:
                _same(m.colors, ref_c)
