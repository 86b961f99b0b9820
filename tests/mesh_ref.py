"""Numpy restatement of the PLY / STL rules (DESIGN.md 7f), written independently of csrc/mesh_loader.cu: the reference
the host loader and the GPU decoder are compared with, plus the vertex-colour shading rule of the rasteriser on top of
the C oracle's triangle-id map."""
from __future__ import annotations

import struct
from pathlib import Path

import numpy as np

_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2", "ushort": "u2",
          "uint16": "u2", "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4", "float": "f4", "float32": "f4",
          "double": "f8", "float64": "f8"}


def _f32(d: float) -> np.float32:
    if d != d:  # NaN: the quiet NaN of its sign
        return np.frombuffer(struct.pack("<I", 0xFFC00000 if np.signbit(d) else 0x7FC00000), np.float32)[0]
    return np.float32(d)


def read_ply(path):
    """(verts f32 (Nv,3), colors u8 (Nv,3) | None, tris i32 (Nt,3))."""
    data = Path(path).read_bytes()
    end = data.index(b"end_header")
    end = data.index(b"\n", end) + 1
    lines = data[:end].decode().split("\n")
    fmt, elems = None, []
    for ln in lines[1:]:
        t = ln.split()
        if not t or t[0] in ("comment", "obj_info", "end_header"):
            continue
        if t[0] == "format":
            fmt = t[1]
        elif t[0] == "element":
            elems.append((t[1], int(t[2]), []))
        elif t[0] == "property":
            elems[-1][2].append(("list", _TYPES[t[2]], _TYPES[t[3]], t[4]) if t[1] == "list" else ("s", _TYPES[t[1]], t[2]))
    body = data[end:]
    if fmt == "ascii":
        tokens = [float(x) for x in body.split()]
        pos = 0

        def take(dt):
            nonlocal pos
            v = tokens[pos]
            pos += 1
            return v if dt[0] == "f" else int(v)
    else:
        e = "<" if fmt == "binary_little_endian" else ">"
        pos = 0

        def take(dt):
            nonlocal pos
            a = np.frombuffer(body, np.dtype(e + dt), 1, pos)[0]
            pos += np.dtype(dt).itemsize
            return a
    verts, cols, tris = None, None, []
    for name, count, props in elems:
        scal = [p[2] for p in props if p[0] == "s"]
        use_col = name == "vertex" and all(c in scal for c in ("red", "green", "blue")) and all(
            p[1] == "u1" for p in props if p[0] == "s" and p[2] in ("red", "green", "blue"))
        if name == "vertex" and verts is None:
            verts = np.zeros((count, 3), np.float32)
            cols = np.zeros((count, 3), np.uint8) if use_col else None
        for r in range(count):
            for p in props:
                if p[0] == "list":
                    n = int(take(p[1]))
                    vals = [int(take(p[2])) for _ in range(n)]
                    if name == "face" and p[3] in ("vertex_indices", "vertex_index"):
                        for k in range(1, n - 1):
                            tris.append((vals[0], vals[k], vals[k + 1]))
                    continue
                v = take(p[1])
                if name == "vertex" and p[2] in ("x", "y", "z"):
                    if fmt != "ascii" and p[1] == "f4":
                        verts[r, "xyz".index(p[2])] = v  # float keeps its bits
                    else:
                        verts[r, "xyz".index(p[2])] = _f32(float(v))
                elif name == "vertex" and cols is not None and p[2] in ("red", "green", "blue"):
                    cols[r, ("red", "green", "blue").index(p[2])] = int(v)
    return verts, cols, np.asarray(tris, np.int32).reshape(-1, 3)


def read_stl_soup(path):
    """(F*3, 3) float32 corners in file order."""
    data = Path(path).read_bytes()
    if len(data) >= 84 and len(data) == 84 + 50 * struct.unpack("<I", data[80:84])[0]:
        n = struct.unpack("<I", data[80:84])[0]
        rec = np.frombuffer(data, np.dtype([("n", "<f4", (3,)), ("v", "<f4", (9,)), ("a", "<u2")]), n, 84)
        return rec["v"].reshape(-1, 3).copy()
    out = []
    for ln in data.decode().splitlines():
        t = ln.split()
        if t and t[0] == "vertex":
            out.append([_f32(float(x)) for x in t[1:4]])
    return np.asarray(out, np.float32).reshape(-1, 3)


def weld(corners):
    """First-occurrence weld: (verts (Nv,3) f32, tris (Nt,3) i32) with degenerate facets dropped."""
    key_of, verts, ids = {}, [], []
    bits = corners.view(np.uint32).copy()
    bits[bits == 0x80000000] = 0  # -0.0 == +0.0
    for i, c in enumerate(corners):
        if np.isnan(c).any():
            ids.append(len(verts))
            verts.append(c)
            continue
        k = tuple(bits[i])
        if k not in key_of:
            key_of[k] = len(verts)
            verts.append(c)
        ids.append(key_of[k])
    ids = np.asarray(ids, np.int32).reshape(-1, 3)
    keep = (ids[:, 0] != ids[:, 1]) & (ids[:, 1] != ids[:, 2]) & (ids[:, 0] != ids[:, 2])
    return np.asarray(verts, np.float32).reshape(-1, 3), ids[keep]


def read_stl(path):
    return weld(read_stl_soup(path))


def _edge(ax, ay, bx, by, cx, cy):
    return (bx - ax) * (cy - ay) - (by - ay) * (cx - ax)


def shade_vertex_colors(verts, tris, colors, rot, tri_map, h, w):
    """(V,H,W,3) uint8 RGB of the vertex-colour rule where tri_map >= 0 (the oracle's triangle ids), 255 elsewhere:
    window coordinates as the rasteriser computes them, fp32 barycentrics, c = (l0*c0 + l1*c1) + l2*c2,
    (int)(c + 0.5) clamped to [0,255].  numpy float32 arithmetic rounds every operation like the --fmad=false kernel."""
    f = np.float32
    out = np.full(tri_map.shape + (3,), 255, np.uint8)
    kx, ky = f(w / 300.0), f(h / 300.0)
    v64 = verts.astype(np.float64)
    for view in range(rot.shape[0]):
        R = rot[view].reshape(9)
        xr = (((R[0] * v64[:, 0] + R[1] * v64[:, 1]) + R[2] * v64[:, 2])).astype(f)
        yr = (((R[3] * v64[:, 0] + R[4] * v64[:, 1]) + R[5] * v64[:, 2])).astype(f)
        sx, sy = (xr + f(150.0)) * kx, (f(150.0) - yr) * ky
        py, px = np.nonzero(tri_map[view] >= 0)
        t = tri_map[view][py, px]
        i0, i1, i2 = tris[t, 0], tris[t, 1], tris[t, 2]
        cx, cy = px.astype(f) + f(0.5), py.astype(f) + f(0.5)
        area = _edge(sx[i0], sy[i0], sx[i1], sy[i1], sx[i2], sy[i2])
        l0 = _edge(sx[i1], sy[i1], sx[i2], sy[i2], cx, cy) / area
        l1 = _edge(sx[i2], sy[i2], sx[i0], sy[i0], cx, cy) / area
        l2 = _edge(sx[i0], sy[i0], sx[i1], sy[i1], cx, cy) / area
        for ch in range(3):
            c = (l0 * colors[i0, ch].astype(f) + l1 * colors[i1, ch].astype(f)) + l2 * colors[i2, ch].astype(f)
            out[view, py, px, ch] = np.clip(c + f(0.5), f(0), f(255)).astype(np.int32)
    return out
