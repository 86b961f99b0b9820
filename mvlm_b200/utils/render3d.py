"""Multi-view renderer: host-side mirror of the reference's ObjVTKRenderer3D
(src/mvlm/utils/render3d.py:12-193) on top of the CUDA rasteriser (csrc/raster.cu).

Same constructor arguments, same methods and return values:
  multiview_render(path) -> (image_stack float32 (V,H,W,4) in [0,1], transform_stack (V,6), mesh)
where `mesh` (an io_obj.Mesh) plays the role of the reference's vtkPolyData.
"""
from __future__ import annotations

import time
from pathlib import Path

import numpy as np
import torch

from .. import ops
from ..io_mesh import check_scan_path, load_mesh
from ..io_obj import Mesh

__all__ = ["ObjRenderer3D", "ObjVTKRenderer3D", "fixed_eight_views", "rotation_matrices"]


def fixed_eight_views() -> np.ndarray:
    """The n_views == 8 preset (render3d.py:93-111): (+-30, +-15/+-45, 0), float32."""
    return np.array([[30, 15, 0, 0, 0, 0], [30, -15, 0, 0, 0, 0], [30, 45, 0, 0, 0, 0], [30, -45, 0, 0, 0, 0],
                     [-30, 15, 0, 0, 0, 0], [-30, -15, 0, 0, 0, 0], [-30, 45, 0, 0, 0, 0], [-30, -45, 0, 0, 0, 0]],
                    dtype=np.float32)


def _rx(a):
    return np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])


def _ry(a):
    return np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])


def _rz(a):
    return np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])


def rotation_matrices(transform_stack: np.ndarray) -> np.ndarray:
    """(V,>=3) [rx, ry, rz] in degrees -> (V,3,3) float64, R = Ry @ Rx @ Rz.

    This is both the renderer's vertex transform (vtkTransform RotateY, RotateX, RotateZ,
    render3d.py:140-145) and the estimator's ray rotation (estimator3d.py:57).  Angles keep the dtype
    of `transform_stack` while np.deg2rad / np.cos / np.sin are evaluated, as in the reference.
    """
    out = np.empty((transform_stack.shape[0], 3, 3), dtype=np.float64)
    for i in range(transform_stack.shape[0]):
        rx, ry, rz = transform_stack[i, :3]
        out[i] = (_ry(np.deg2rad(ry)) @ _rx(np.deg2rad(rx))) @ _rz(np.deg2rad(rz))
    return out


_PARALLEL_COPY_BYTES = 4 << 20
_COPY_THREADS = 4
_pool = None


def _copy_pool():
    global _pool
    if _pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _pool = ThreadPoolExecutor(_COPY_THREADS, thread_name_prefix="mvlm-stage")
    return _pool


class _PinnedStage:
    """One slot of the renderer's upload ring: page-locked host buffers the four arrays of a scan are copied into, so
    that the host -> device transfer is asynchronous whatever memory the caller's arrays live in (a pageable source
    makes cudaMemcpyAsync stall the enqueueing thread behind the work already in the stream: measured 39 instead of
    51 scans/s with two scans in flight)."""

    def __init__(self):
        self.buf = {}
        self.done = None  # CUDA event recorded after the slot's last transfer

    def stage(self, name: str, a: np.ndarray) -> torch.Tensor:
        flat = a.reshape(-1)
        b = self.buf.get(name)
        if b is None or b.dtype != torch.from_numpy(flat[:0].copy()).dtype or b.numel() < flat.size:
            b = torch.empty((max(flat.size, 1),), dtype=torch.from_numpy(flat[:0].copy()).dtype, pin_memory=True)
            self.buf[name] = b
        view = b[:flat.size]
        dst = view.numpy()
        if flat.nbytes < _PARALLEL_COPY_BYTES:
            np.copyto(dst, flat)
        else:  # multi-million-triangle scans: one core copies ~6 GB/s, the copy loop releases the GIL
            edges = np.linspace(0, flat.size, _COPY_THREADS + 1).astype(np.int64)
            list(_copy_pool().map(lambda i: np.copyto(dst[edges[i]:edges[i + 1]], flat[edges[i]:edges[i + 1]]),
                                  range(_COPY_THREADS)))
        return view.view(a.shape)


def page_table(pages) -> np.ndarray:
    """(3P,) int32: texel offset, height and width of every page in the packed RGBA texels of
    DeviceMesh.raster_input."""
    table, off = [], 0
    for p in pages:
        table += [off, p.shape[0], p.shape[1]]
        off += p.shape[0] * p.shape[1]
    return np.asarray(table, dtype=np.int32)


def _on_current_stream(a: torch.Tensor, ready) -> torch.Tensor:
    """A device-side array of a scan (decoded or parsed on a loader's side stream) for use on the current stream."""
    if ready is not None:
        torch.cuda.current_stream().wait_event(ready)
    if a.is_cuda:
        a.record_stream(torch.cuda.current_stream())  # keep its memory until the current stream is done with it
    return a


class DeviceMesh:
    """Device-resident copy of a Mesh (uploaded once per scan): `arrays` maps the names of Mesh.arrays to device
    tensors; verts, tris, uvs, tex, colors, tri_page, pages and page_table name them (None when absent)."""

    def __init__(self, mesh: Mesh, device: torch.device, stage: _PinnedStage | None = None):
        def up(name, a, ready):
            if isinstance(a, torch.Tensor):  # decoded (nvJPEG) or parsed (parser="gpu") on the loader's side stream
                return _on_current_stream(a, ready)
            a = np.ascontiguousarray(a)
            if device.type != "cuda":
                return torch.from_numpy(a.copy()).to(device)
            t = torch.from_numpy(a) if a.flags.writeable else None
            if t is not None and t.is_pinned():
                return t.to(device, non_blocking=True)       # caller's arrays are page-locked already
            if stage is None:
                return torch.from_numpy(a.copy()).to(device)
            return stage.stage(name, a).to(device, non_blocking=True)

        if stage is not None and stage.done is not None:
            stage.done.synchronize()                          # the slot's previous transfer has left the host buffers
        arrays = {name: up(name, a, ready) for name, a, ready in mesh.arrays()}
        if stage is not None and device.type == "cuda":
            stage.done = torch.cuda.Event()
            stage.done.record()
        self._wrap(mesh, arrays)

    @classmethod
    def from_device(cls, mesh: Mesh, arrays: dict) -> "DeviceMesh":
        """Wraps the device tensors of Mesh.arrays, by name (sharding.upload_mesh_sharded)."""
        self = cls.__new__(cls)
        self._wrap(mesh, arrays)
        return self

    def _wrap(self, mesh: Mesh, arrays: dict) -> None:
        self.mesh, self.arrays = mesh, arrays
        self.verts, self.tris, self.uvs, self.tex, self.colors, self.tri_page, self.page_table = \
            (arrays.get(k) for k in ("verts", "tris", "uvs", "tex", "colors", "tri_page", "page_table"))
        self.pages = None if mesh.pages is None else [arrays[f"page{i}"] for i in range(len(mesh.pages))]

    def raster_input(self) -> ops.RasterInput:
        """The scan as ops.raster_multiscan reads it, built once per device mesh: the texture as RGBA (tex4), the
        vertex colours as (Nv,4) RGBA (one 4-byte load per texel or vertex in the rasteriser), and for a scan with
        pages, the RGBA texels of all pages packed into one (1, N, 4) u8 buffer (offsets in page_table) as the texture
        with the int32 (Nt + 3P,) table: the page of every triangle, then page_table."""
        r = self.__dict__.get("_raster_input")
        if r is None:
            tex, table = self.tex4(), None
            if self.pages is not None:
                tex = torch.empty((1, sum(p.shape[0] * p.shape[1] for p in self.pages), 4), dtype=torch.uint8,
                                  device=self.tri_page.device)
                tex[..., 3] = 255
                off = 0
                for p in self.pages:
                    n = p.shape[0] * p.shape[1]
                    tex[0, off:off + n, :3] = p.reshape(n, 3)
                    off += n
                table = torch.cat([self.tri_page.reshape(-1), self.page_table])
            colors = None
            if self.colors is not None:
                colors = torch.empty((self.colors.shape[0], 4), dtype=torch.uint8, device=self.colors.device)
                colors[:, :3] = self.colors
                colors[:, 3] = 255
            r = self._raster_input = ops.RasterInput(self.verts, self.uvs, self.tris, tex, colors, table)
        return r

    def paged(self):
        """(packed RGBA texels of all pages, int32 (Nt + 3P,) table) of raster_input, or (None, None) without pages."""
        r = self.raster_input()
        return (None, None) if r.pages is None else (r.tex, r.pages)

    def tex4(self):
        """The texture as RGBA (one 4-byte load per texel in the rasteriser), expanded once per device mesh."""
        if self.tex is None:
            return None
        t = self.__dict__.get("_tex4")
        if t is None:
            if self.tex.shape[-1] == 4:
                t = self.tex
            else:
                t = torch.empty(self.tex.shape[:2] + (4,), dtype=torch.uint8, device=self.tex.device)
                t[..., :3] = self.tex
                t[..., 3] = 255
            self._tex4 = t
        return t

    def snap_grid(self):
        """Spatial index for the surface snap, built at most once per device mesh (None below ops.SNAP_GRID_MIN_TRIS,
        where the brute-force scan is faster than building the grid)."""
        if "_snap_grid" not in self.__dict__:
            self._snap_grid = ops.SnapGrid(self.verts, self.tris) if self.tris.shape[0] >= ops.SNAP_GRID_MIN_TRIS else None
        return self._snap_grid

    @property
    def h2d_bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.arrays.values())


class ObjRenderer3D:
    def __init__(self, n_views: int = 8, image_size: tuple = (256, 256), offscreen: bool = True,
                 min_x_angle: int = -40, max_x_angle: int = 40, min_y_angle: int = -80, max_y_angle: int = 80,
                 min_z_angle: int = -20, max_z_angle: int = 20, min_scale: float = 1.4, max_scale: float = 1.9,
                 min_tx: int = -20, max_tx: int = 20, min_ty: int = -20, max_ty: int = 20,
                 channel_mode: str = "RGB+depth", device: str = "cuda"):
        self.n_views = n_views
        self.image_size = image_size
        self.pre_align = None       # set by the pipeline (seam path only; the fused path transforms before upload)
        self.last_pre_align = None
        self.offscreen = offscreen  # kept for signature compatibility; there is no window
        self.min_x_angle, self.max_x_angle = min_x_angle, max_x_angle
        self.min_y_angle, self.max_y_angle = min_y_angle, max_y_angle
        self.min_z_angle, self.max_z_angle = min_z_angle, max_z_angle
        self.min_scale, self.max_scale = min_scale, max_scale
        self.min_tx, self.max_tx = min_tx, max_tx
        self.min_ty, self.max_ty = min_ty, max_ty
        self.channel_mode = channel_mode
        self.device = torch.device(device)
        self.slack = 5
        self.side_length = max([150 - (-150), 150 - (-150)]) * 1.0 / 2
        # injected view list (tests / benchmarks); None -> generate like the reference
        self.transforms: np.ndarray | None = None
        self.verbose = True
        # suffixes multiview_render accepts (set by the pipeline's scan_formats)
        self.scan_formats = ("obj",)
        # where multiview_render finds an OBJ's texture (set by the pipeline's texture_source)
        self.texture_source = "stem"

    # render3d.py:79-89 (GLOBAL np.random, same draw order)
    def random_transform(self, size=1):
        rx = np.random.randint(self.min_x_angle, self.max_x_angle, size=size)
        ry = np.random.randint(self.min_y_angle, self.max_y_angle, size=size)
        rz = np.random.randint(self.min_z_angle, self.max_z_angle, size=size)
        scale = np.random.uniform(self.min_scale, self.max_scale, size=size)
        tx = np.random.randint(self.min_tx, self.max_tx, size=size)
        ty = np.random.randint(self.min_ty, self.max_ty, size=size)
        return np.stack((rx, ry, rz, scale, tx, ty), axis=1)

    # render3d.py:92-112
    def generate_3d_transformations(self):
        if self.transforms is not None:
            return np.asarray(self.transforms)
        if self.n_views == 8:
            return fixed_eight_views()
        return self.random_transform(size=self.n_views)

    def upload(self, mesh: Mesh) -> DeviceMesh:
        """Asynchronous host -> device copy of a scan on the current stream (through a ring of pinned staging slots
        unless the caller's arrays are page-locked already).  A dedicated copy stream was measured and dropped: with two
        scans in flight the 5 MB upload is 0.1 ms of an 18 ms scan (53.3 -> 53.5 scans/s on one GPU, 431.6 -> 429.8 on
        eight; profiles/r1_experiments.txt)."""
        if self.device.type != "cuda":
            return DeviceMesh(mesh, self.device)
        if not hasattr(self, "_stages"):
            self._stages = [_PinnedStage() for _ in range(4)]
            self._stage_i = 0
        st = self._stages[self._stage_i % len(self._stages)]
        self._stage_i += 1
        return DeviceMesh(mesh, self.device, st)

    def reserve_upload_slots(self, n: int) -> None:
        """At least `n` pinned staging slots: the batch drivers keep up to (scans per pass) x (passes in flight + 1)
        scans between their upload and the end of their transfer, and a slot reused sooner makes the host wait for
        the transfer of an earlier pass."""
        if self.device.type != "cuda":
            return
        if not hasattr(self, "_stages"):
            self._stages = [_PinnedStage() for _ in range(4)]
            self._stage_i = 0
        self._stages += [_PinnedStage() for _ in range(n - len(self._stages))]

    def rotations_device(self, transform_stack: np.ndarray) -> torch.Tensor:
        """(V,9) float64 device tensor of R = Ry@Rx@Rz per view; cached for the last transform stack
        (the per-view numpy evaluation that mirrors the reference dtype flow costs ~20 us per view)."""
        key = (transform_stack.dtype.str, transform_stack.shape, transform_stack.tobytes())
        if getattr(self, "_rot_key", None) != key:
            self._rot = torch.from_numpy(rotation_matrices(transform_stack).reshape(-1, 9)).to(self.device)
            self._rot_key = key
        return self._rot

    def render_device(self, dmesh: DeviceMesh, transform_stack: np.ndarray, want_f32=False, want_tri=False, want_z=False):
        """All views in one launch pair; returns the dict of device tensors of ops.raster_multiview."""
        return self.render_pass([dmesh], [transform_stack], want_f32=want_f32, want_tri=want_tri, want_z=want_z)

    def render_pass(self, dmeshes: list, transform_stacks: list, want_f32=False, want_tri=False, want_z=False,
                    reserve_views: int = 0):
        """The views of several scans in one launch sequence (ops.raster_multiscan), scan-major; every scan's images
        equal render_device's.  `reserve_views`: the persistent image is sized for at least this many views (the
        pass size the batch driver plans), so that a shorter pass uses a prefix of it at the same address."""
        rot = self.rotations_device(np.concatenate([np.asarray(t) for t in transform_stacks]))
        h, w = self.image_size[0], self.image_size[1]
        total = rot.shape[0]
        # persistent z-buffer / u8 image (overwritten by the next render): stable pointers let the CNN replay
        # its CUDA graph, and no allocation happens per scan
        if getattr(self, "_buf_key", None) != (h, w) or self._u8.shape[0] < total:
            self._u8 = torch.empty((max(total, reserve_views), h, w, 4), dtype=torch.uint8, device=self.device)
            self._zbuf = None
            self._buf_key = (h, w)
        # the rasteriser's scratch also holds the per-(view, vertex) window coordinates: it grows with the largest scan
        max_nv = max(d.verts.shape[0] for d in dmeshes)
        lib = ops._lib.load()
        need = lib.mvlm_raster_multiscan_workspace_bytes(len(dmeshes), total // len(dmeshes), h, w, max_nv)
        if self._zbuf is None or self._zbuf.numel() * 8 < need:
            n = lib.mvlm_raster_multiscan_workspace_bytes(len(dmeshes), total // len(dmeshes), h, w, int(max_nv * 1.25))
            self._zbuf = torch.empty(((n + 7) // 8,), dtype=torch.int64, device=self.device)
        return ops.raster_multiscan([d.raster_input() for d in dmeshes], rot, h, w, self.channel_mode,
                                    want_f32=want_f32, want_tri=want_tri, want_z=want_z, zbuf=self._zbuf,
                                    out_u8=self._u8[:total])

    # render3d.py:114-177
    def render_3d_multi_rgb_geometry_depth(self, transform_stack, file_name):
        tt = time.time()
        mesh = file_name if isinstance(file_name, Mesh) else load_mesh(file_name, texture_source=self.texture_source)
        if self.pre_align is not None:  # legacy "pre-align" block, see utils/prealign.py; the seam path's back-transform
            import dataclasses           # is Pipeline._predict_seams'

            from . import prealign

            self.last_pre_align = prealign.affine(mesh.verts, self.pre_align)
            mesh = dataclasses.replace(mesh, verts=prealign.apply(mesh.verts, *self.last_pre_align))
        dmesh = self.upload(mesh)
        if self.verbose:
            print("Render [1] - Setup time: ", f"{time.time() - tt:08.6f} s")
        tt = time.time()
        out = self.render_device(dmesh, np.asarray(transform_stack), want_f32=True)
        image_stack = out["f32"].cpu().numpy()
        if self.verbose:
            print("Render [2] - Render", f"{time.time() - tt:08.6f} s")
        return image_stack, mesh

    # render3d.py:179-193
    def multiview_render(self, file_name: Path):
        t = time.time()
        file_name = Path(file_name)
        if not file_name.exists():
            raise FileNotFoundError(f"File {file_name} does not exist")
        check_scan_path(file_name, self.scan_formats)
        if self.verbose:
            print("Render [0] - Prepare", f"{time.time() - t:08.6f} s")
        transformation_stack = self.generate_3d_transformations()
        image_stack, mesh = self.render_3d_multi_rgb_geometry_depth(transformation_stack, file_name)
        # the kernel already writes u8/255 in float32 (render3d.py:191)
        return image_stack, transformation_stack, mesh


# drop-in name of the reference class
ObjVTKRenderer3D = ObjRenderer3D
