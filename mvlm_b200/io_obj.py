"""Scan loader: Wavefront OBJ (+ optional `<stem>.jpg` texture) -> flat arrays.

Replaces vtkOBJReader / vtkJPEGReader as used by the reference's obj_to_actor
(src/mvlm/utils/utils3d.py:10-36): positions `v`, texture coordinates `vt`, faces
`f a[/b[/c]] ...` (polygons are fan-triangulated).  Like vtkOBJReader, a position that is
referenced with different `vt` indices is duplicated so that every output vertex has exactly
one (position, uv) pair.

texture_source="mtl" (our extension, DESIGN.md 7g) textures a scan from its MTL materials instead: `mtllib` /
`usemtl` in the OBJ, `newmtl` / `map_Kd` in the libraries, one texture page per distinct file (Mesh.pages) and the
page of every triangle (Mesh.tri_page).
"""
from __future__ import annotations

import os
from dataclasses import dataclass, replace
from pathlib import Path

import numpy as np


@dataclass
class Mesh:
    verts: object              # (Nv,3) float32: numpy array, or a CUDA tensor (parser="gpu")
    tris: object               # (Nt,3) int32: numpy array, or a CUDA tensor (parser="gpu")
    uvs: object | None         # (Nv,2) float32: numpy array, or a CUDA tensor (parser="gpu")
    texture: object | None     # (Th,Tw,3) uint8, row 0 = top of the image: numpy array, or a CUDA tensor (nvJPEG decode)
    path: Path | None = None
    texture_ready: object | None = None  # CUDA event recorded after a device-side decode (texture is a CUDA tensor)
    geometry_ready: object | None = None  # CUDA event recorded after a device-side parse (verts / uvs / tris are CUDA tensors)
    colors: object | None = None  # (Nv,3) uint8 per-vertex RGB (PLY scans, io_mesh): numpy array, or a CUDA tensor
    # texture_source="mtl" with more than one page (texture is then None): (Th_p,Tw_p,3) uint8 pages, row 0 = top
    # (numpy arrays, or CUDA tensors behind texture_ready), and the (Nt,) int32 page of every triangle (-1 = white)
    pages: list | None = None
    tri_page: object | None = None

    @property
    def bbox_diagonal(self) -> float:
        return float(np.linalg.norm(self.verts.max(0) - self.verts.min(0)))

    def arrays(self) -> list:
        """(name, array, ready event) of every array of the scan that is present, in upload order: verts, tris, uvs,
        tex, colors, tri_page, page0 .. page{P-1} and page_table (render3d.page_table, computed from the pages).  A
        CUDA tensor is read only after its event: texture_ready for the texture and the pages, geometry_ready for the
        rest.  The names key the pinned staging buffers of the uploads, which are reused from scan to scan."""
        g, t = self.geometry_ready, self.texture_ready
        out = [("verts", self.verts, g), ("tris", self.tris, g), ("uvs", self.uvs, g), ("tex", self.texture, t),
               ("colors", self.colors, g), ("tri_page", self.tri_page, g)]
        if self.pages is not None:
            from .utils.render3d import page_table

            out += [(f"page{i}", p, t) for i, p in enumerate(self.pages)] + [("page_table", page_table(self.pages), g)]
        return [e for e in out if e[1] is not None]


def _texture_file(path: Path):
    """`<stem>.jpg` next to the scan (utils3d.py:26); FLAME models (`flame*.obj`) use `mean_texture.jpg` of their folder
    instead (utils3d.py:39-51).  Returns None when there is no texture file."""
    if path.name.startswith("flame"):
        print("Loading flame texture")
        jpg = path.parent / "mean_texture.jpg"
        if not jpg.exists():
            print("Could not load flame texture", jpg)
            return None
        return jpg
    jpg = path.with_suffix(".jpg")
    return jpg if jpg.exists() else None


def _read_image(file: Path):
    """(Th,Tw,3) uint8 through PIL, or None for a missing or unreadable file."""
    try:
        from PIL import Image

        return np.asarray(Image.open(file).convert("RGB"), dtype=np.uint8)
    except Exception:  # noqa: BLE001 - same policy as the reference: ignore an unreadable texture
        return None


TEXTURE_DECODERS = ("pil", "nvjpeg")


def _check_texture_decoder(texture_decoder: str) -> None:
    if texture_decoder not in TEXTURE_DECODERS:
        raise ValueError(f"Unknown texture decoder: {texture_decoder}")


def _read_texture(file: Path, texture_decoder: str, device):
    """One image file -> ((Th,Tw,3) uint8, event recorded after a device-side decode or None), or (None, None) when it
    is missing or unreadable.  JPEG files under texture_decoder="nvjpeg" are decoded on the GPU (a CUDA tensor),
    everything else through PIL (a numpy array)."""
    _check_texture_decoder(texture_decoder)
    if texture_decoder == "nvjpeg" and file.suffix.lower() in (".jpg", ".jpeg"):
        return _decode_jpeg_nvjpeg(file, device)
    return _read_image(file), None


def _load_texture(path: Path, texture_decoder: str = "pil", device=None):
    """The `<stem>.jpg` rule (_texture_file) through _read_texture: (texture, event | None)."""
    _check_texture_decoder(texture_decoder)  # also for a scan without a texture file
    jpg = _texture_file(path)
    return (None, None) if jpg is None else _read_texture(jpg, texture_decoder, device)


TEXTURE_SOURCES = ("stem", "mtl")


def check_texture_source(texture_source: str) -> str:
    if texture_source not in TEXTURE_SOURCES:
        raise ValueError(f"Unknown texture source: {texture_source} (supported: {', '.join(TEXTURE_SOURCES)})")
    return texture_source


def _text(b: bytes) -> str:
    return b.decode("utf-8", "surrogateescape")


def _relative(folder: Path, name: str) -> Path:
    return folder / name.replace("\\", "/")


def parse_mtl(path: Path, materials: dict) -> None:
    """Adds the materials of one MTL library to `materials` (name -> texture file, or None without `map_Kd`).
    `newmtl <name>`: the rest of the line, trimmed; a name defined before keeps its first definition.  `map_Kd ...
    <file>`: the last whitespace-separated token, relative to the library's folder (`\\` is a separator), options before
    it ignored.  Statements may be indented; every other statement is ignored.  Raises OSError for an unreadable file."""
    current = None
    for raw in path.read_bytes().split(b"\n"):
        line = raw.strip(b" \t\r")
        if line.startswith((b"newmtl ", b"newmtl\t")):
            name = _text(line[7:].strip(b" \t\r"))
            current = None if name in materials else name
            if current is not None:
                materials[current] = None
        elif current is not None and line.startswith((b"map_Kd ", b"map_Kd\t")):
            tokens = line[7:].split()
            if tokens:
                materials[current] = _relative(path.parent, _text(tokens[-1]))


_tls = None


def loader_state(device):
    """Per-thread state of the device-side loaders: a side stream on `device` (the loader threads of
    Pipeline.predict_files parse and decode on it while the main stream computes), and the buffers of the GPU parser,
    which grow to the largest file the thread has read."""
    import threading

    import torch

    global _tls
    if _tls is None:
        _tls = threading.local()
    device = torch.device(device)
    if getattr(_tls, "stream", None) is None or _tls.device != device:
        _tls.stream, _tls.device = torch.cuda.Stream(device), device
        _tls.pinned = _tls.text = _tls.workspace = None
    return _tls


def _grown(st, name: str, n: int, **alloc):
    """The loader state's uint8 buffer `name` (pinned, text, workspace), reallocated with max(n, 1) bytes when it holds
    fewer than n.  The old buffer is dropped first, so that a large file can reuse its memory."""
    import torch

    if getattr(st, name) is None or getattr(st, name).numel() < n:
        setattr(st, name, None)
        setattr(st, name, torch.empty((max(n, 1),), dtype=torch.uint8, **alloc))
    return getattr(st, name)


def decode_on_device(device, ws_bytes: int, info, phase1, phase2):
    """Runs a two-phase device decoder (csrc/obj_parse.cu, csrc/mesh_parse.cu) on the calling thread's side stream.
    phase1(workspace, stream) fills `info` and returns the status (it synchronises the side stream; the main stream
    never waits); phase2(workspace, stream) allocates and writes the outputs.  Returns phase2's tuple + (event behind
    the outputs,), None on info.fallback (the host loader reads the file), or raises ValueError when phase 1 fails."""
    import torch

    from . import _lib

    device = torch.device(device)
    st = loader_state(device)
    with torch.cuda.device(device), torch.cuda.stream(st.stream):
        ws = _grown(st, "workspace", ws_bytes, device=device).data_ptr()
        if phase1(ws, st.stream.cuda_stream) != 0:
            raise ValueError(_lib.load().mvlm_last_error().decode("utf-8", "replace"))
        if info.fallback:
            return None
        out = phase2(ws, st.stream.cuda_stream)
        ready = torch.cuda.Event(enable_timing=True)
        ready.record(st.stream)
    return out + (ready,)


def _decode_jpeg_nvjpeg(jpg: Path, device):
    """One JPEG file -> (Th,Tw,3) uint8 CUDA tensor + the event recorded behind the decode, or (None, None) when it is
    missing or unreadable (mvlm_jpeg_decode_rgb on a per-thread side stream: the loader threads of
    Pipeline.predict_files decode while the main stream computes)."""
    import torch

    from . import _lib

    try:
        data = jpg.read_bytes()
    except OSError:
        return None, None
    lib = _lib.load()
    import ctypes as C

    w, h = C.c_int(), C.c_int()
    if lib.mvlm_jpeg_info(data, len(data), C.byref(w), C.byref(h)) != 0:
        return None, None  # same policy as the reference: ignore an unreadable texture
    device = torch.device(device)
    _tls = loader_state(device)
    with torch.cuda.device(device), torch.cuda.stream(_tls.stream):
        tex = torch.empty((h.value, w.value, 3), dtype=torch.uint8, device=device)
        if lib.mvlm_jpeg_decode_rgb(data, len(data), tex.data_ptr(), w.value, h.value, _tls.stream.cuda_stream) != 0:
            return None, None
        ready = torch.cuda.Event()
        ready.record(_tls.stream)
    return tex, ready


def read_pinned(path: Path, device):
    """The bytes of `path` in the calling thread's page-locked buffer (grown to the largest file read): a uint8 tensor
    view of exactly the file's size."""
    n = path.stat().st_size
    pinned = _grown(loader_state(device), "pinned", n, pin_memory=True)
    view = memoryview(pinned.numpy())[:n]
    got = 0
    with open(path, "rb", buffering=0) as fh:
        while got < n:
            k = fh.readinto(view[got:])
            if not k:
                break
            got += k
    if got != n:
        raise ValueError(f"mvlm_obj_load: short read on {path}")
    return pinned[:n]


def parse_obj_device(text, path: Path, device):
    """Runs csrc/obj_parse.cu on the file's bytes `text` (uint8 CUDA tensor) on the calling thread's side stream:
    returns (verts, uvs | None, tris, event recorded after the arrays are written) as CUDA tensors, or None when the
    file must be parsed on the host (a number of more than 19 significant digits, or beyond the parser's capacity).
    Raises ValueError with the host parser's message for a bad file."""
    parsed = _parse_device(text, path, device)
    return None if parsed is None else parsed[:4]


def _parse_device(text, path: Path, device, materials: bool = False):
    """parse_obj_device; with `materials` (MVLM_OBJ_MATERIALS) the fifth element is (info, name lines) for
    _with_device_materials, else None."""
    import ctypes as C

    import torch

    from . import _lib

    lib = _lib.load()
    n = text.numel()
    flags = _lib.OBJ_MATERIALS if materials else 0
    ws_bytes = lib.mvlm_obj_parse_workspace_bytes_ex(n, flags)
    if ws_bytes == 0:
        return None
    info, lines, n_lines = _lib.ObjParseInfo(), None, C.c_int()
    if materials:
        st = loader_state(device)
        if getattr(st, "name_lines", None) is None:
            st.name_lines = (_lib.ObjNameLine * _lib.OBJ_MAX_NAME_LINES)()
        lines = st.name_lines

    def outputs(ws, stream):
        verts = torch.empty((info.n_verts, 3), dtype=torch.float32, device=device)
        tris = torch.empty((info.n_tris, 3), dtype=torch.int32, device=device)
        uvs = torch.empty((info.n_verts, 2), dtype=torch.float32, device=device) if info.has_uv else None
        _lib.check(lib.mvlm_obj_parse_write(C.byref(info), ws, verts.data_ptr(),
                                            None if uvs is None else uvs.data_ptr(), tris.data_ptr(), stream),
                   "mvlm_obj_parse_write")
        return verts, uvs, tris

    parsed = decode_on_device(device, ws_bytes, info, lambda ws, stream: lib.mvlm_obj_parse_device_ex(
        text.data_ptr(), n, str(path).encode(), ws, ws_bytes, flags, stream, C.byref(info), lines,
        _lib.OBJ_MAX_NAME_LINES if materials else 0, C.byref(n_lines)), outputs)
    if parsed is None:
        return None
    extra = (info, [(lines[i].offset, lines[i].kind, lines[i].tris_before) for i in range(n_lines.value)]) \
        if materials else None
    return parsed + (extra,)


def _load_geometry_gpu(path: Path, device, materials: bool = False):
    """parser="gpu": the file is read into page-locked memory, copied to the device on the side stream (the previous
    file's copy is complete: the first phase of its parse synchronised that stream) and parsed there."""
    import torch

    from . import _lib

    if _lib.load().mvlm_obj_parse_workspace_bytes_ex(path.stat().st_size, _lib.OBJ_MATERIALS if materials else 0) == 0:
        return None  # beyond the parser's capacity
    device = torch.device(device)
    host = read_pinned(path, device)
    st = loader_state(device)
    with torch.cuda.device(device), torch.cuda.stream(st.stream):
        text = _grown(st, "text", host.numel(), device=device)[:host.numel()]
        text.copy_(host, non_blocking=True)
    parsed = _parse_device(text, path, device, materials)
    if parsed is None or not materials:
        return parsed
    return parsed[:4] + ((parsed[4][0], _name_lines(host.numpy(), parsed[4][1])),)


def _name_lines(data: np.ndarray, lines: list):
    """(kind, name, triangles before) of the name lines the GPU parser found, the names read from the file's bytes:
    the rest of the line, trimmed, like the host loader."""
    out = []
    for off, kind, before in lines:
        end, step = off, 256
        while True:
            nl = np.flatnonzero(data[end:end + step] == 10)
            if nl.size or end + step >= data.size:
                end = end + int(nl[0]) if nl.size else data.size
                break
            end, step = end + step, step * 4
        out.append((kind, _text(data[off + 7:end].tobytes().strip(b" \t\r")), before))
    return out


def _load_pages(path: Path, order: list, names: list, libraries: list, texture_decoder: str, device):
    """texture_source="mtl": (pages, page of every material (len(names) + 1 entries, the last -1 for "no material"),
    event behind the last device-side decode or None), or None when the scan has no usable page.  `order`: the
    materials in order of first use by a triangle; pages are the distinct resolved texture files in that order, and a
    file that is missing or unreadable is reported once and its triangles stay white."""
    materials = {}
    for name in libraries:
        lib_path = _relative(path.parent, name)
        try:
            parse_mtl(lib_path, materials)
        except OSError:
            print("Could not load material library", lib_path)
    page_of = np.full(len(names) + 1, -1, np.int32)  # [-1] (the last slot) stays -1: triangles without a material
    by_file, pages, ready = {}, [], None
    for m in order:
        file = materials.get(names[m])
        if file is None:
            continue
        key = os.path.normpath(file)
        if key not in by_file:
            img, ev = _read_texture(file, texture_decoder, device)
            if img is None:
                print("Could not load texture", file)
                by_file[key] = -1
            else:
                by_file[key] = len(pages)
                pages.append(img)
                ready = ev if ev is not None else ready
        page_of[m] = by_file[key]
    if not pages:
        return None
    return pages, page_of, ready


def _paged_mesh(mesh: Mesh, pages: list, one_page: bool, tri_page, ready, geometry_ready) -> Mesh:
    """A scan whose triangles all use one page (`one_page`) is an ordinary single-texture scan."""
    if one_page:
        return replace(mesh, texture=pages[0], texture_ready=ready)
    return replace(mesh, texture_ready=ready, geometry_ready=geometry_ready, pages=pages, tri_page=tri_page)


def _with_materials(mesh: Mesh, materials, texture_decoder: str, device) -> Mesh | None:
    """The scan textured from its MTL materials (host loader: per-triangle material, names, libraries), or None when
    the `<stem>.jpg` rule applies (no usable page)."""
    tm, names, libraries = materials
    # materials in order of first use: the first triangle of every run of equal ordinals, then first occurrences
    starts = np.flatnonzero(np.concatenate(([True], tm[1:] != tm[:-1]))) if tm.size else np.zeros(0, np.int64)
    order = list(dict.fromkeys(int(m) for m in tm[starts] if m >= 0))
    paged = _load_pages(mesh.path, order, names, libraries, texture_decoder, device)
    if paged is None:
        return None
    pages, page_of, ready = paged
    tri_page = page_of[tm]
    return _paged_mesh(mesh, pages, len(pages) == 1 and (tri_page == 0).all(), tri_page, ready, mesh.geometry_ready)


def _with_device_materials(mesh: Mesh, info, lines: list, texture_decoder: str, device) -> Mesh | None:
    """_with_materials for a scan parsed on the GPU: the material of every `usemtl` ordinal comes from the name lines,
    and mvlm_obj_parse_tri_page writes the page of every triangle on the loader's side stream."""
    import ctypes as C

    import torch

    from . import _lib

    libraries = [name for kind, name, _ in lines if kind == 2]
    usemtl = [(name, before) for kind, name, before in lines if kind == 1]
    ids, names, line_id = {}, [], []
    for name, _ in usemtl:
        line_id.append(ids.setdefault(name, len(ids)))
        if len(names) < len(ids):
            names.append(name)
    n_tris = info.n_tris
    ends = [before for _, before in usemtl[1:]] + [n_tris]
    used = [end > before for (_, before), end in zip(usemtl, ends)]  # the line has faces after it
    order = list(dict.fromkeys(m for m, u in zip(line_id, used) if u))
    paged = _load_pages(mesh.path, order, names, libraries, texture_decoder, device)
    if paged is None:
        return None
    pages, page_of, ready = paged
    line_page = np.ascontiguousarray(page_of[np.asarray(line_id, np.int64)] if line_id else np.zeros(0), np.int32)
    unassigned = not usemtl or usemtl[0][1] > 0  # triangles before the first usemtl
    one_page = len(pages) == 1 and not unassigned and all(p == 0 for p, u in zip(line_page, used) if u)
    if one_page:
        return _paged_mesh(mesh, pages, True, None, ready, None)
    lib = _lib.load()
    device = torch.device(device)
    st = loader_state(device)
    with torch.cuda.device(device), torch.cuda.stream(st.stream):
        tri_page = torch.empty((n_tris,), dtype=torch.int32, device=device)
        _lib.check(lib.mvlm_obj_parse_tri_page(C.byref(info), st.workspace.data_ptr(), line_page.ctypes.data,
                                               len(line_page), tri_page.data_ptr(), st.stream.cuda_stream),
                   "mvlm_obj_parse_tri_page")
        geometry_ready = torch.cuda.Event(enable_timing=True)
        geometry_ready.record(st.stream)
    return _paged_mesh(mesh, pages, False, tri_page, ready, geometry_ready)


def load_obj(path: Path | str, load_texture: bool = True, n_threads: int = 0, texture_decoder: str = "pil",
             device="cuda", parser: str = "host", texture_source: str = "stem") -> Mesh:
    """Native loader: what the pipeline uses.
    parser: "host" (csrc/obj_loader.cu through the C-ABI, multi-threaded parse; numpy arrays) or "gpu"
    (csrc/obj_parse.cu: the same arrays bit for bit and the same errors, parsed on `device` from the file's bytes;
    verts / uvs / tris are CUDA tensors written on the loader thread's side stream, and Mesh.geometry_ready is the
    event behind them.  A file with a number of more than 19 significant digits is parsed on the host: numpy arrays.)
    texture_decoder: "pil" (host decode, libjpeg-turbo: the decoder the parity tests share with the oracle) or
    "nvjpeg" (csrc/jpeg_decode.cu: decoded on the GPU into device memory; values may differ by a few LSB).
    texture_source: "stem" (the reference's `<stem>.jpg` / `mean_texture.jpg` rule) or "mtl" (the scan's MTL
    materials, DESIGN.md 7g: JPEG pages through texture_decoder, other formats through PIL; the `<stem>.jpg` rule when
    no page is usable); with parser="gpu" the device parser finds the material lines too."""
    import ctypes as C

    from . import _lib

    path = Path(path)
    if not path.is_file():
        raise ValueError(f"File {path} does not exist.")
    if parser not in ("host", "gpu"):
        raise ValueError(f"Unknown OBJ parser: {parser}")
    check_texture_source(texture_source)
    materials = texture_source == "mtl" and load_texture
    if parser == "gpu":
        parsed = _load_geometry_gpu(path, device, materials)
        if parsed is not None:
            verts, uvs, tris, geometry_ready = parsed[:4]
            if materials and uvs is not None and parsed[4][1]:
                mesh = Mesh(verts=verts, tris=tris, uvs=uvs, texture=None, path=path, geometry_ready=geometry_ready)
                textured = _with_device_materials(mesh, *parsed[4], texture_decoder, device)
                if textured is not None:
                    return textured
            texture, ready = _load_texture(path, texture_decoder, device) if load_texture and uvs is not None \
                else (None, None)
            return Mesh(verts=verts, tris=tris, uvs=uvs, texture=texture, path=path, texture_ready=ready,
                        geometry_ready=geometry_ready)
    lib = _lib.load()
    h = C.c_void_p()
    if materials:
        rc = lib.mvlm_obj_load_ex(str(path).encode(), n_threads, _lib.OBJ_MATERIALS, C.byref(h))
    else:
        rc = lib.mvlm_obj_load(str(path).encode(), n_threads, C.byref(h))
    if rc != 0:
        raise ValueError(lib.mvlm_last_error().decode("utf-8", "replace"))
    try:
        nv, nt, has_uv = C.c_int(), C.c_int(), C.c_int()
        _lib.check(lib.mvlm_obj_counts(h, C.byref(nv), C.byref(nt), C.byref(has_uv)), "mvlm_obj_counts")
        verts = np.empty((nv.value, 3), dtype=np.float32)
        tris = np.empty((nt.value, 3), dtype=np.int32)
        uvs = np.empty((nv.value, 2), dtype=np.float32) if has_uv.value else None
        _lib.check(lib.mvlm_obj_copy(h, verts.ctypes.data, None if uvs is None else uvs.ctypes.data, tris.ctypes.data),
                   "mvlm_obj_copy")
        if materials:
            tri_material = np.empty((nt.value,), dtype=np.int32)
            n_mat, n_lib = C.c_int(), C.c_int()
            _lib.check(lib.mvlm_obj_materials(h, tri_material.ctypes.data, C.byref(n_mat), C.byref(n_lib)),
                       "mvlm_obj_materials")
            names = [_text(lib.mvlm_obj_material_name(h, i)) for i in range(n_mat.value)]
            libraries = [_text(lib.mvlm_obj_library_name(h, i)) for i in range(n_lib.value)]
    finally:
        lib.mvlm_obj_free(h)
    mesh = Mesh(verts=verts, tris=tris, uvs=uvs, texture=None, path=path)
    if materials and uvs is not None:
        textured = _with_materials(mesh, (tri_material, names, libraries), texture_decoder, device)
        if textured is not None:
            return textured
    if load_texture and uvs is not None:
        mesh.texture, mesh.texture_ready = _load_texture(path, texture_decoder, device)
    return mesh
