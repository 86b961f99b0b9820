"""Seeded synthetic inputs: a textured face-like mesh (OBJ + JPG, OBJ + MTL pages, PLY, STL), view transforms, ray sets.

The reference's sample scans are missing blobs (.MISSING_LARGE_BLOBS) and there is no network,
so every benchmark and parity test runs on these (SURVEY.md section 8d).
"""
from __future__ import annotations

from pathlib import Path

import numpy as np


def face_mesh(grid: int = 224, seed: int = 1234):
    """Height-field 'face': grid x grid vertices on an ellipsoidal cap (+-90 x +-110 mm, ~80 mm deep)
    with seeded low-frequency bumps, centred so that it stays inside the +-150 mm orthographic
    window for every view angle the renderer draws.  Returns (verts f32 (N,3), uvs f32 (N,2),
    tris i32 (T,3))."""
    rng = np.random.RandomState(seed)
    a = np.linspace(-1.0, 1.0, grid)
    aa, bb = np.meshgrid(a, a, indexing="xy")
    r2 = (aa ** 2 + bb ** 2) / 2.0
    z = 80.0 * np.sqrt(np.clip(1.0 - r2, 0.0, 1.0))
    # nose / brow / chin style bumps
    for _ in range(6):
        cx, cy = rng.uniform(-0.5, 0.5, 2)
        s = rng.uniform(0.08, 0.3)
        amp = rng.uniform(-6.0, 14.0)
        z += amp * np.exp(-((aa - cx) ** 2 + (bb - cy) ** 2) / (2 * s * s))
    z += 18.0 * np.exp(-((aa) ** 2 + (bb + 0.05) ** 2) / (2 * 0.12 ** 2))  # nose
    x = 90.0 * aa
    y = 110.0 * bb
    verts = np.stack([x, y, z], -1).reshape(-1, 3)
    verts -= verts.mean(0, keepdims=True)
    # keep inside the 150 mm view sphere
    rmax = np.linalg.norm(verts, axis=1).max()
    if rmax > 145.0:
        verts *= 145.0 / rmax
    u = (aa + 1.0) / 2.0
    v = (bb + 1.0) / 2.0
    uvs = np.stack([u, v], -1).reshape(-1, 2)
    idx = np.arange(grid * grid).reshape(grid, grid)
    q00, q01, q10, q11 = idx[:-1, :-1], idx[:-1, 1:], idx[1:, :-1], idx[1:, 1:]
    t1 = np.stack([q00, q01, q11], -1).reshape(-1, 3)
    t2 = np.stack([q00, q11, q10], -1).reshape(-1, 3)
    tris = np.concatenate([t1, t2], 0)
    return verts.astype(np.float32), uvs.astype(np.float32), tris.astype(np.int32)


def face_texture(size: int = 1024, seed: int = 1234) -> np.ndarray:
    """(size,size,3) uint8: smooth seeded colour noise plus high-contrast markers."""
    rng = np.random.RandomState(seed + 1)
    t = np.linspace(0, 1, size, dtype=np.float32)
    xx, yy = np.meshgrid(t, t, indexing="xy")
    img = np.zeros((size, size, 3), np.float32)
    for c in range(3):
        acc = np.zeros((size, size), np.float32)
        for _ in range(5):
            fx, fy = rng.uniform(1, 9, 2)
            ph = rng.uniform(0, 2 * np.pi)
            acc += np.sin(2 * np.pi * (fx * xx + fy * yy) + ph).astype(np.float32)
        img[..., c] = 0.55 + 0.12 * acc
    for _ in range(40):
        cx, cy = rng.uniform(0.05, 0.95, 2)
        r = rng.uniform(0.004, 0.02)
        col = rng.uniform(0, 1, 3)
        m = (xx - cx) ** 2 + (yy - cy) ** 2 < r * r
        img[m] = col
    return (np.clip(img, 0, 1) * 255).astype(np.uint8)


def write_obj(path: Path, verts, uvs, tris, texture: np.ndarray | None = None, jpeg_quality: int = 95) -> Path:
    """Writes `<path>.obj` (v / vt / f a/a b/b c/c) and, if given, `<stem>.jpg` beside it
    (the file the reference's obj_to_actor looks for, src/mvlm/utils/utils3d.py:26)."""
    path = Path(path)
    with open(path, "w") as f:
        f.write("# mvlm_b200 synthetic scan\n")
        np.savetxt(f, verts, fmt="v %.6f %.6f %.6f")
        if uvs is not None:
            np.savetxt(f, uvs, fmt="vt %.6f %.6f")
            t = tris + 1
            np.savetxt(f, np.stack([t[:, 0], t[:, 0], t[:, 1], t[:, 1], t[:, 2], t[:, 2]], 1), fmt="f %d/%d %d/%d %d/%d")
        else:
            np.savetxt(f, tris + 1, fmt="f %d %d %d")
    if texture is not None:
        from PIL import Image

        Image.fromarray(texture).save(path.with_suffix(".jpg"), quality=jpeg_quality)
    return path


def write_obj_mtl(path: Path, verts, uvs, tris, pages: list, tri_page, formats=None, jpeg_quality: int = 95) -> Path:
    """Writes an OBJ scan textured through MTL materials (DESIGN.md 7g): `<path>.obj` with `mtllib <stem>.mtl`, its
    faces in file order split into `usemtl` groups wherever `tri_page` changes, `<stem>.mtl` with one material per page
    (`map_Kd <stem>_<i>.<format>`) and one without a texture for page -1, and the pages themselves.
    pages: (Th,Tw,3) uint8 images of any sizes; tri_page: (Nt,) page of every triangle (-1: the untextured material);
    formats: file format per page, "jpg" (default) or "png"."""
    from PIL import Image

    path = Path(path)
    tri_page = np.asarray(tri_page)
    formats = formats or ["jpg"] * len(pages)
    files = [f"{path.stem}_{i}.{fmt}" for i, fmt in enumerate(formats)]
    for img, fmt, name in zip(pages, formats, files):
        Image.fromarray(img).save(path.parent / name, **({"quality": jpeg_quality} if fmt == "jpg" else {}))
    lines = []
    for i, name in enumerate(files):
        lines += [f"newmtl page{i}", "Ka 1 1 1", "Kd 1 1 1", f"map_Kd {name}", ""]
    lines += ["newmtl untextured", "Kd 1 1 1", ""]
    path.with_suffix(".mtl").write_text("\n".join(lines))
    t = np.asarray(tris) + 1
    cuts = np.flatnonzero(np.diff(tri_page)) + 1
    with open(path, "w") as f:
        f.write(f"# mvlm_b200 synthetic scan\nmtllib {path.stem}.mtl\n")
        np.savetxt(f, verts, fmt="v %.6f %.6f %.6f")
        np.savetxt(f, uvs, fmt="vt %.6f %.6f")
        for lo, hi in zip(np.concatenate(([0], cuts)), np.concatenate((cuts, [len(t)]))):
            f.write(f"usemtl {'untextured' if tri_page[lo] < 0 else f'page{tri_page[lo]}'}\n")
            tt = t[lo:hi]
            np.savetxt(f, np.stack([tt[:, 0], tt[:, 0], tt[:, 1], tt[:, 1], tt[:, 2], tt[:, 2]], 1),
                       fmt="f %d/%d %d/%d %d/%d")
    return path


_PLY_NUMPY = {"char": "i1", "uchar": "u1", "short": "i2", "ushort": "u2", "int": "i4", "uint": "u4", "float": "f4",
              "double": "f8", "int8": "i1", "uint8": "u1", "int16": "i2", "uint16": "u2", "int32": "i4", "uint32": "u4",
              "float32": "f4", "float64": "f8"}


def write_ply(path: Path, verts, faces, colors=None, fmt: str = "binary_little_endian", pos_type: str = "float",
              count_type: str = "uchar", index_type: str = "int") -> Path:
    """Writes a PLY scan: `vertex` x y z of `pos_type` (+ uchar red green blue when `colors` (Nv,3) uint8 is given) and
    `face` vertex_indices lists.  faces: (F,3) int array, or a list of index sequences (polygons of any length).
    fmt: "ascii", "binary_little_endian" or "binary_big_endian"."""
    path = Path(path)
    verts = np.asarray(verts)
    polys = [list(map(int, f)) for f in faces]
    end = {"binary_little_endian": "<", "binary_big_endian": ">", "ascii": "<"}[fmt]
    head = ["ply", f"format {fmt} 1.0", "comment mvlm_b200 synthetic scan", f"element vertex {len(verts)}",
            f"property {pos_type} x", f"property {pos_type} y", f"property {pos_type} z"]
    if colors is not None:
        head += ["property uchar red", "property uchar green", "property uchar blue"]
    head += [f"element face {len(polys)}", f"property list {count_type} {index_type} vertex_indices", "end_header"]
    with open(path, "wb") as f:
        f.write(("\n".join(head) + "\n").encode())
        if fmt == "ascii":
            pos = verts.astype(_PLY_NUMPY[pos_type])
            for i in range(len(verts)):
                row = [repr(float(x)) if pos.dtype.kind == "f" else str(int(x)) for x in pos[i]]
                if colors is not None:
                    row += [str(int(c)) for c in colors[i]]
                f.write((" ".join(row) + "\n").encode())
            for p in polys:
                f.write((" ".join(map(str, [len(p)] + p)) + "\n").encode())
            return path
        fields = [(c, end + _PLY_NUMPY[pos_type]) for c in "xyz"]
        if colors is not None:
            fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
        rec = np.empty(len(verts), dtype=fields)
        for k, c in enumerate("xyz"):
            rec[c] = verts[:, k]
        if colors is not None:
            for k, c in enumerate(("red", "green", "blue")):
                rec[c] = np.asarray(colors)[:, k]
        f.write(rec.tobytes())
        cdt, idt = np.dtype(end + _PLY_NUMPY[count_type]), np.dtype(end + _PLY_NUMPY[index_type])
        if all(len(p) == 3 for p in polys):  # one record array for the usual all-triangle file
            frec = np.empty(len(polys), dtype=[("n", cdt), ("i", idt, (3,))])
            frec["n"] = 3
            frec["i"] = np.asarray(polys, dtype=np.int64).reshape(-1, 3)
            f.write(frec.tobytes())
        else:
            for p in polys:
                f.write(np.array([len(p)], cdt).tobytes() + np.array(p, idt).tobytes())
    return path


def write_stl(path: Path, verts, tris, binary: bool = True, header: bytes = b"mvlm_b200 synthetic scan") -> Path:
    """Writes an STL triangle soup (three corners per facet, facet normals zero): binary (80-byte `header`, count,
    50-byte records) or ASCII (`solid` ... `endsolid`, coordinates printed with repr, which round-trips float32
    through float64)."""
    path = Path(path)
    corners = np.asarray(verts, np.float32)[np.asarray(tris, np.int64)]  # (F,3,3)
    if binary:
        rec = np.zeros(len(corners), dtype=[("n", "<f4", (3,)), ("v", "<f4", (9,)), ("a", "<u2")])
        rec["v"] = corners.reshape(-1, 9)
        with open(path, "wb") as f:
            f.write(header[:80].ljust(80, b" "))
            f.write(np.array([len(corners)], "<u4").tobytes())
            f.write(rec.tobytes())
        return path
    lines = ["solid synthetic"]
    for c in corners:
        lines += ["facet normal 0 0 0", "  outer loop"]
        lines += [f"    vertex {float(x)!r} {float(y)!r} {float(z)!r}" for x, y, z in c]
        lines += ["  endloop", "endfacet"]
    lines.append("endsolid synthetic")
    Path(path).write_text("\n".join(lines) + "\n")
    return path


def random_view_transforms(n_views: int, seed: int | None = None) -> np.ndarray:
    """The reference's ObjVTKRenderer3D.random_transform draw order (src/mvlm/utils/render3d.py:79-89):
    rx in [-40,40), ry in [-80,80), rz in [-20,20) integers, then the unused scale/tx/ty draws;
    (V,6) float64.  `seed` seeds the GLOBAL numpy RNG exactly like a harness around the reference would."""
    if seed is not None:
        np.random.seed(seed)
    rx = np.random.randint(-40, 40, size=n_views)
    ry = np.random.randint(-80, 80, size=n_views)
    rz = np.random.randint(-20, 20, size=n_views)
    scale = np.random.uniform(1.4, 1.9, size=n_views)
    tx = np.random.randint(-20, 20, size=n_views)
    ty = np.random.randint(-20, 20, size=n_views)
    return np.stack((rx, ry, rz, scale, tx, ty), axis=1)


def synthetic_rays(n_landmarks: int = 84, n_views: int = 200, outlier_frac: float = 0.3, seed: int = 1234):
    """Consensus micro-benchmark input (BASELINE.json config 5): per landmark a true 3D point,
    V rays through it (0.5 mm jitter), `outlier_frac` of them displaced by U(-80,80) mm.
    Returns (peaks (L,V,3) f32 [row, col, value], starts, ends (L,V,3) f64, truth (L,3))."""
    rng = np.random.RandomState(seed)
    truth = rng.uniform(-80, 80, (n_landmarks, 3))
    ang = np.deg2rad(np.stack([rng.randint(-40, 40, n_views), rng.randint(-80, 80, n_views),
                               rng.randint(-20, 20, n_views)], 1).astype(np.float64))
    starts = np.empty((n_landmarks, n_views, 3))
    ends = np.empty((n_landmarks, n_views, 3))
    for v in range(n_views):
        ax, ay, az = ang[v]
        mx = np.array([[1, 0, 0], [0, np.cos(ax), -np.sin(ax)], [0, np.sin(ax), np.cos(ax)]])
        my = np.array([[np.cos(ay), 0, np.sin(ay)], [0, 1, 0], [-np.sin(ay), 0, np.cos(ay)]])
        mz = np.array([[np.cos(az), -np.sin(az), 0], [np.sin(az), np.cos(az), 0], [0, 0, 1]])
        r = my @ mx @ mz
        cam = truth @ r.T  # camera coordinates of the points
        cam = cam + rng.normal(0, 0.5, cam.shape)
        out = rng.uniform(0, 1, n_landmarks) < outlier_frac
        cam[out, :2] += rng.uniform(-80, 80, (int(out.sum()), 2))
        s = np.stack([cam[:, 0], cam[:, 1], np.full(n_landmarks, 500.0)], 1)
        e = np.stack([cam[:, 0], cam[:, 1], np.full(n_landmarks, -500.0)], 1)
        starts[:, v] = s @ r
        ends[:, v] = e @ r
    peaks = np.zeros((n_landmarks, n_views, 3), np.float32)
    peaks[:, :, 2] = rng.uniform(0, 1, (n_landmarks, n_views)).astype(np.float32)
    return peaks, starts, ends, truth


def hypothesis_table(n_landmarks: int, n_hyp: int, seed: int = 1234) -> np.ndarray:
    """Shared seeded RANSAC draws (L,H,8) uint32; line index = draw mod n_lines_after_filter."""
    return np.random.RandomState(seed).randint(0, 2 ** 32, (n_landmarks, n_hyp, 8), dtype=np.uint64).astype(np.uint32)
