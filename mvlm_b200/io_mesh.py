"""Scan loader for every supported format: Wavefront OBJ (io_obj.load_obj, unchanged), PLY and STL.

PLY (ascii / binary little or big endian) gives positions, triangles and, when the vertex element has uchar
red / green / blue, per-vertex colours (Mesh.colors); STL (ascii / binary) is a triangle soup whose corners are welded
into shared vertices.  Neither has texture coordinates.  The rules are DESIGN.md 7f; csrc/mesh_loader.cu is their
specification and csrc/mesh_parse.cu decodes binary files on the GPU with the same result, bit for bit.
"""
from __future__ import annotations

from pathlib import Path

import numpy as np

from .io_obj import Mesh, check_texture_source, decode_on_device, load_obj, read_pinned

SUFFIXES = {"obj": ".obj", "ply": ".ply", "stl": ".stl"}


def check_scan_formats(scan_formats) -> tuple:
    """Validated tuple of enabled format names ("obj", "ply", "stl")."""
    formats = tuple(scan_formats)
    for f in formats:
        if f not in SUFFIXES:
            raise ValueError(f"Unknown scan format: {f} (supported: {', '.join(SUFFIXES)})")
    if not formats:
        raise ValueError("scan_formats must name at least one format")
    return formats


def is_scan_file(path: Path, scan_formats) -> bool:
    """Whether `path` has the suffix of an enabled format: `.obj` exactly (the OBJ-only pipeline's check), `.ply` /
    `.stl` in any case."""
    if path.suffix == ".obj":
        return "obj" in scan_formats
    suffix = path.suffix.lower()
    return suffix in (".ply", ".stl") and suffix[1:] in scan_formats


def check_scan_file(path: Path, scan_formats) -> None:
    """Raises the pipeline's error for a file that is not of an enabled format.  With the default ("obj",) the message
    is the one the OBJ-only pipeline has always raised."""
    if is_scan_file(path, scan_formats):
        return
    if tuple(scan_formats) == ("obj",):
        raise ValueError(f"File {path} is not an .obj file. Only .obj files are supported.")
    names = ", ".join(SUFFIXES[f] for f in scan_formats)
    raise ValueError(f"File {path} is not a scan file. Only {names} files are supported.")


def check_scan_path(path: Path, scan_formats) -> None:
    """check_scan_file for an existing path that is about to be loaded, after a FileNotFoundError when it is not a
    regular file.  A missing path is the caller's to handle."""
    if not path.is_file():
        raise FileNotFoundError(f"File {path} is not a file")
    check_scan_file(path, scan_formats)


def parse_mesh_device(path: Path, device):
    """parser="gpu" for a PLY / STL file: the bytes are read into the calling thread's page-locked buffer and decoded
    by csrc/mesh_parse.cu on the thread's side stream.  Returns (verts, colors | None, tris, event recorded after the
    arrays are written) as CUDA tensors, or None when the file must be read on the host (ASCII, faces that are not all
    triangles, an index out of range, beyond the decoder's capacity).  Raises ValueError for a bad PLY header."""
    import ctypes as C

    import torch

    from . import _lib

    lib = _lib.load()
    is_stl = 1 if path.suffix.lower() == ".stl" else 0
    n = path.stat().st_size
    ws_bytes = lib.mvlm_mesh_parse_workspace_bytes(n, is_stl)
    if ws_bytes == 0:
        return None
    host = read_pinned(path, device)
    info = _lib.MeshParseInfo()

    def outputs(ws, stream):
        verts = torch.empty((info.n_verts, 3), dtype=torch.float32, device=device)
        tris = torch.empty((info.n_tris, 3), dtype=torch.int32, device=device)
        colors = torch.empty((info.n_verts, 3), dtype=torch.uint8, device=device) if info.has_colors else None
        _lib.check(lib.mvlm_mesh_parse_write(C.byref(info), ws, verts.data_ptr(),
                                             None if colors is None else colors.data_ptr(), tris.data_ptr(), stream),
                   "mvlm_mesh_parse_write")
        return verts, colors, tris

    # once phase 1 returns (it synchronises the side stream), the page-locked buffer is free for the next file
    return decode_on_device(device, ws_bytes, info, lambda ws, stream: lib.mvlm_mesh_parse_device(
        host.data_ptr(), n, is_stl, str(path).encode(), ws, ws_bytes, stream, C.byref(info)), outputs)


def load_ply_stl(path: Path | str, n_threads: int = 0, device="cuda", parser: str = "host") -> Mesh:
    """PLY / STL scan -> Mesh(verts, tris, uvs=None, texture=None, colors).
    parser: "host" (csrc/mesh_loader.cu through the C-ABI; numpy arrays) or "gpu" (csrc/mesh_parse.cu: the same arrays
    bit for bit, CUDA tensors written on the loader thread's side stream behind Mesh.geometry_ready; files the decoder
    does not take are read on the host: numpy arrays)."""
    import ctypes as C

    from . import _lib

    path = Path(path)
    if not path.is_file():
        raise ValueError(f"File {path} does not exist.")
    if parser not in ("host", "gpu"):
        raise ValueError(f"Unknown scan parser: {parser}")
    if parser == "gpu":
        parsed = parse_mesh_device(path, device)
        if parsed is not None:
            verts, colors, tris, ready = parsed
            return Mesh(verts=verts, tris=tris, uvs=None, texture=None, path=path, geometry_ready=ready, colors=colors)
    lib = _lib.load()
    h = C.c_void_p()
    if lib.mvlm_mesh_load(str(path).encode(), n_threads, C.byref(h)) != 0:
        raise ValueError(lib.mvlm_last_error().decode("utf-8", "replace"))
    try:
        nv, nt, has_colors = C.c_int(), C.c_int(), C.c_int()
        _lib.check(lib.mvlm_mesh_counts(h, C.byref(nv), C.byref(nt), C.byref(has_colors)), "mvlm_mesh_counts")
        verts = np.empty((nv.value, 3), dtype=np.float32)
        tris = np.empty((nt.value, 3), dtype=np.int32)
        colors = np.empty((nv.value, 3), dtype=np.uint8) if has_colors.value else None
        _lib.check(lib.mvlm_mesh_copy(h, verts.ctypes.data, None if colors is None else colors.ctypes.data,
                                      tris.ctypes.data), "mvlm_mesh_copy")
    finally:
        lib.mvlm_mesh_free(h)
    return Mesh(verts=verts, tris=tris, uvs=None, texture=None, path=path, colors=colors)


def load_mesh(path: Path | str, load_texture: bool = True, n_threads: int = 0, texture_decoder: str = "pil",
              device="cuda", parser: str = "host", texture_source: str = "stem") -> Mesh:
    """Any supported scan by its suffix: `.obj` -> io_obj.load_obj (all arguments apply), `.ply` / `.stl` (any case)
    -> load_ply_stl (no texture: load_texture, texture_decoder and texture_source do not apply)."""
    path = Path(path)
    suffix = path.suffix.lower()
    check_texture_source(texture_source)
    if path.suffix == ".obj":
        return load_obj(path, load_texture=load_texture, n_threads=n_threads, texture_decoder=texture_decoder,
                        device=device, parser=parser, texture_source=texture_source)
    if suffix in (".ply", ".stl"):
        return load_ply_stl(path, n_threads=n_threads, device=device, parser=parser)
    raise ValueError(f"File {path} is not an .obj, .ply or .stl file.")
