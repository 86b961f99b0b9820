"""Pure numpy restatement of the scan loader (oracle: test infrastructure only, see oracle/__init__.py).

Checker of the native parser mvlm_b200/csrc/obj_loader.cu (mvlm_obj_load): same semantics as vtkOBJReader as used by
the reference's obj_to_actor (src/mvlm/utils/utils3d.py:16-21) -- `v` / `vt` / `f a[/b[/c]]` with 1-based or negative
relative indices, polygons fan-triangulated, one output vertex per distinct (position, vt) pair in ascending order.
"""
from __future__ import annotations

from pathlib import Path

import numpy as np

from mvlm_b200.io_obj import Mesh, _load_texture


def load_obj_python(path: Path | str, load_texture: bool = True) -> Mesh:
    """Pure numpy restatement of the same loader: test infrastructure (the checker of the native parser)."""
    path = Path(path)
    if not path.is_file():
        raise ValueError(f"File {path} does not exist.")
    v_rows, vt_rows, f_rows = [], [], []
    n_v = n_vt = 0
    with open(path, "r", errors="replace") as fh:
        for line in fh:
            if line.startswith("v "):
                v_rows.append(line[2:])
                n_v += 1
            elif line.startswith("vt "):
                vt_rows.append(line[3:])
                n_vt += 1
            elif line.startswith("f "):
                f_rows.append((line[2:], n_v, n_vt))  # counts so far: negative indices are relative to them
    if len(v_rows) == 0:
        raise ValueError(f"File {path} does not contain any points.")
    pos = np.loadtxt(v_rows, dtype=np.float64, ndmin=2, usecols=(0, 1, 2)).astype(np.float32)
    tex = np.loadtxt(vt_rows, dtype=np.float64, ndmin=2, usecols=(0, 1)).astype(np.float32) if vt_rows else None
    corners_v, corners_t = [], []
    for row, v_seen, vt_seen in f_rows:
        toks = row.split()
        vi, ti = [], []
        for tok in toks:
            parts = tok.split("/")
            a = int(parts[0])
            vi.append(a - 1 if a > 0 else v_seen + a)
            if len(parts) > 1 and parts[1] != "":
                b = int(parts[1])
                ti.append(b - 1 if b > 0 else vt_seen + b)
            else:
                ti.append(-1)
        for k in range(1, len(vi) - 1):
            corners_v.append((vi[0], vi[k], vi[k + 1]))
            corners_t.append((ti[0], ti[k], ti[k + 1]))
    cv = np.asarray(corners_v, dtype=np.int64).reshape(-1, 3)
    ct = np.asarray(corners_t, dtype=np.int64).reshape(-1, 3)
    if tex is None or (ct < 0).all():
        verts, uvs, tris = pos, None, cv.astype(np.int32)
    else:
        # unique (position, uv) pairs -> output vertices
        pairs = np.stack([cv.reshape(-1), ct.reshape(-1)], 1)
        uniq, inv = np.unique(pairs, axis=0, return_inverse=True)
        verts = pos[uniq[:, 0]]
        uvs = np.where(uniq[:, 1:2] >= 0, tex[np.clip(uniq[:, 1], 0, None)], 0.0).astype(np.float32)
        tris = inv.reshape(-1, 3).astype(np.int32)
    texture = _load_texture(path)[0] if (load_texture and uvs is not None) else None
    return Mesh(verts=np.ascontiguousarray(verts), tris=np.ascontiguousarray(tris),
                uvs=None if uvs is None else np.ascontiguousarray(uvs), texture=texture, path=path)
