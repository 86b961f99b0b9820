"""Scan loader: Wavefront OBJ (+ optional `<stem>.jpg` texture) -> flat arrays.

Replaces vtkOBJReader / vtkJPEGReader as used by the reference's obj_to_actor
(src/mvlm/utils/utils3d.py:10-36): positions `v`, texture coordinates `vt`, faces
`f a[/b[/c]] ...` (polygons are fan-triangulated).  Like vtkOBJReader, a position that is
referenced with different `vt` indices is duplicated so that every output vertex has exactly
one (position, uv) pair.
"""
from __future__ import annotations

from dataclasses import dataclass
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

    @property
    def bbox_diagonal(self) -> float:
        return float(np.linalg.norm(self.verts.max(0) - self.verts.min(0)))


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


def _load_texture(path: Path):
    jpg = _texture_file(path)
    if jpg is None:
        return None
    try:
        from PIL import Image

        return np.asarray(Image.open(jpg).convert("RGB"), dtype=np.uint8)
    except Exception:  # noqa: BLE001 - same policy as the reference: ignore an unreadable texture
        return None


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


def _decode_texture_nvjpeg(path: Path, device):
    """`<stem>.jpg` -> (Th,Tw,3) uint8 CUDA tensor + the event recorded behind the decode (mvlm_jpeg_decode_rgb on a
    per-thread side stream: the loader threads of Pipeline.predict_files decode while the main stream computes)."""
    import torch

    from . import _lib

    jpg = _texture_file(path)
    if jpg is None:
        return None, None
    data = jpg.read_bytes()
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
    import torch

    st = loader_state(device)
    n = path.stat().st_size
    if st.pinned is None or st.pinned.numel() < n:
        st.pinned = None
        st.pinned = torch.empty((max(n, 1),), dtype=torch.uint8, pin_memory=True)
    view = memoryview(st.pinned.numpy())[:n]
    got = 0
    with open(path, "rb", buffering=0) as fh:
        while got < n:
            k = fh.readinto(view[got:])
            if not k:
                break
            got += k
    if got != n:
        raise ValueError(f"mvlm_obj_load: short read on {path}")
    return st.pinned[:n]


def parse_obj_device(text, path: Path, device):
    """Runs csrc/obj_parse.cu on the file's bytes `text` (uint8 CUDA tensor) on the calling thread's side stream:
    returns (verts, uvs | None, tris, event recorded after the arrays are written) as CUDA tensors, or None when the
    file must be parsed on the host (a number of more than 19 significant digits, or beyond the parser's capacity).
    Raises ValueError with the host parser's message for a bad file."""
    import ctypes as C

    import torch

    from . import _lib

    lib = _lib.load()
    device = torch.device(device)
    st = loader_state(device)
    n = text.numel()
    ws_bytes = lib.mvlm_obj_parse_workspace_bytes(n)
    if ws_bytes == 0:
        return None
    with torch.cuda.device(device), torch.cuda.stream(st.stream):
        if st.workspace is None or st.workspace.numel() < ws_bytes:
            st.workspace = None
            st.workspace = torch.empty((ws_bytes,), dtype=torch.uint8, device=device)
        info = _lib.ObjParseInfo()
        # synchronises the side stream (the sizes of the outputs come back to the host); the main stream never waits
        if lib.mvlm_obj_parse_device(text.data_ptr(), n, str(path).encode(), st.workspace.data_ptr(), ws_bytes,
                                     st.stream.cuda_stream, C.byref(info)) != 0:
            raise ValueError(lib.mvlm_last_error().decode("utf-8", "replace"))
        if info.fallback:
            return None
        verts = torch.empty((info.n_verts, 3), dtype=torch.float32, device=device)
        tris = torch.empty((info.n_tris, 3), dtype=torch.int32, device=device)
        uvs = torch.empty((info.n_verts, 2), dtype=torch.float32, device=device) if info.has_uv else None
        _lib.check(lib.mvlm_obj_parse_write(C.byref(info), st.workspace.data_ptr(), verts.data_ptr(),
                                            None if uvs is None else uvs.data_ptr(), tris.data_ptr(),
                                            st.stream.cuda_stream), "mvlm_obj_parse_write")
        ready = torch.cuda.Event(enable_timing=True)
        ready.record(st.stream)
    return verts, uvs, tris, ready


def _load_geometry_gpu(path: Path, device):
    """parser="gpu": the file is read into page-locked memory, copied to the device on the side stream (the previous
    file's copy is complete: the first phase of its parse synchronised that stream) and parsed there."""
    import torch

    from . import _lib

    if _lib.load().mvlm_obj_parse_workspace_bytes(path.stat().st_size) == 0:
        return None  # beyond the parser's capacity
    device = torch.device(device)
    host = read_pinned(path, device)
    st = loader_state(device)
    with torch.cuda.device(device), torch.cuda.stream(st.stream):
        n = host.numel()
        if st.text is None or st.text.numel() < n:
            st.text = None
            st.text = torch.empty((max(n, 1),), dtype=torch.uint8, device=device)
        text = st.text[:n]
        text.copy_(host, non_blocking=True)
    return parse_obj_device(text, path, device)


def load_obj(path: Path | str, load_texture: bool = True, n_threads: int = 0, texture_decoder: str = "pil",
             device="cuda", parser: str = "host") -> Mesh:
    """Native loader: what the pipeline uses.
    parser: "host" (csrc/obj_loader.cu through the C-ABI, multi-threaded parse; numpy arrays) or "gpu"
    (csrc/obj_parse.cu: the same arrays bit for bit and the same errors, parsed on `device` from the file's bytes;
    verts / uvs / tris are CUDA tensors written on the loader thread's side stream, and Mesh.geometry_ready is the
    event behind them.  A file with a number of more than 19 significant digits is parsed on the host: numpy arrays.)
    texture_decoder: "pil" (host decode, libjpeg-turbo: the decoder the parity tests share with the oracle) or
    "nvjpeg" (csrc/jpeg_decode.cu: decoded on the GPU into device memory; values may differ by a few LSB)."""
    import ctypes as C

    from . import _lib

    path = Path(path)
    if not path.is_file():
        raise ValueError(f"File {path} does not exist.")
    if parser not in ("host", "gpu"):
        raise ValueError(f"Unknown OBJ parser: {parser}")
    if parser == "gpu":
        parsed = _load_geometry_gpu(path, device)
        if parsed is not None:
            verts, uvs, tris, geometry_ready = parsed
            texture, ready = _load_texture_as(path, texture_decoder, device) if load_texture and uvs is not None \
                else (None, None)
            return Mesh(verts=verts, tris=tris, uvs=uvs, texture=texture, path=path, texture_ready=ready,
                        geometry_ready=geometry_ready)
    lib = _lib.load()
    h = C.c_void_p()
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
    finally:
        lib.mvlm_obj_free(h)
    texture, ready = _load_texture_as(path, texture_decoder, device) if load_texture and uvs is not None else (None, None)
    return Mesh(verts=verts, tris=tris, uvs=uvs, texture=texture, path=path, texture_ready=ready)


def _load_texture_as(path: Path, texture_decoder: str, device):
    """(texture, event recorded after a device-side decode or None)."""
    if texture_decoder == "nvjpeg":
        return _decode_texture_nvjpeg(path, device)
    if texture_decoder == "pil":
        return _load_texture(path), None
    raise ValueError(f"Unknown texture decoder: {texture_decoder}")
