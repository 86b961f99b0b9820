"""Numpy restatement of the OBJ material rules (DESIGN.md 7g): the checker of mvlm_obj_load_ex's MVLM_OBJ_MATERIALS
output (csrc/obj_loader.cu) and of the paged texel rule of csrc/raster.cu."""
from __future__ import annotations

import re
from pathlib import Path

import numpy as np

_BLANKS = re.compile(rb"[ \t\r]+")


def obj_materials(path: Path | str):
    """(tri_material (Nt,) int32, distinct usemtl names in order of first appearance, mtllib names): a triangle takes
    the name of the last `usemtl` line before its `f` line (-1 before the first); lines end at '\\n' only."""
    names, ids, libraries, tri = [], {}, [], []
    current = -1
    for line in Path(path).read_bytes().split(b"\n"):
        if line.startswith(b"f "):
            corners = [t for t in _BLANKS.split(line[2:]) if t]
            tri += [current] * max(len(corners) - 2, 0)
        elif line.startswith((b"usemtl ", b"usemtl\t")):
            name = line[7:].strip(b" \t\r").decode("utf-8", "surrogateescape")
            if name not in ids:
                ids[name] = len(names)
                names.append(name)
            current = ids[name]
        elif line.startswith((b"mtllib ", b"mtllib\t")):
            libraries.append(line[7:].strip(b" \t\r").decode("utf-8", "surrogateescape"))
    return np.asarray(tri, dtype=np.int32), names, libraries


def paged_image(images: list, tri: np.ndarray, tri_page: np.ndarray, background: np.ndarray) -> np.ndarray:
    """Image of a paged scan from one render per page (`images[p]`: the scan rendered with page p as its only
    texture): each covered pixel takes the render of its triangle's page, or `background` (the untextured render:
    white) for page -1; uncovered pixels are the same in every render."""
    out = background.copy()
    hit = tri >= 0
    page = np.full(tri.shape, -1, np.int64)
    page[hit] = tri_page[tri[hit]]
    for p, img in enumerate(images):
        m = page == p
        out[m] = img[m]
    return out
