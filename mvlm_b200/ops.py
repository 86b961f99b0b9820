"""Thin Python wrappers over single C-ABI stage calls (used by tests and the host classes).

Tensors are torch CUDA tensors used purely as device buffers.
"""
from __future__ import annotations

import contextlib
import ctypes as C

import os
from typing import NamedTuple

import torch

from . import _lib
from ._lib import ConvArgs, check, cur_stream, ptr


def pack_conv_weight(w_oihw: torch.Tensor, cout_pad: int, cin_pad: int) -> torch.Tensor:
    """fp32 OIHW (cuda) -> bf16 [cout_pad, kw, kh, cin_pad] (cuda)."""
    lib = _lib.load()
    w = w_oihw.contiguous().float()
    cout, cin, kh, kw = w.shape
    out = torch.empty((cout_pad, kw, kh, cin_pad), dtype=torch.bfloat16, device=w.device)
    check(lib.mvlm_pack_conv_weight(ptr(w), cout, cin, kh, kw, cout_pad, cin_pad, ptr(out), cur_stream()),
          "mvlm_pack_conv_weight")
    return out


def conv2d_bf16(x: torch.Tensor, wpacked: torch.Tensor, *, cin: int | None = None, n_tile: int,
                kh: int = 3, kw: int = 3, y_off0: int | None = None, x_off0: int | None = None,
                bias=None, mid=None, pre=None, res1=None, res2=None, out_raw=None, post=None,
                out_f32=None, argmax_keys=None, cout_real: int | None = None,
                up=(1, 1, 0, 0), pool2: bool = False, res_up=None) -> None:
    """One fused conv launch.

    x          : (N,H,W,Cs) bf16; the first `cin` channels are read.
    pre / post : (scale f32[cout_pad], shift f32[cout_pad], out bf16 (N,H,W,Cs'), channel offset)
    res1/res2  : (tensor bf16 (N,H,W,Cs'), channel offset)
    res_up     : (tensor bf16 (N,H/2,W/2,Cs'), channel offset), added with nearest x2 up-sampling
    out_raw    : (tensor bf16 (N,H,W,Cs'), channel offset)
    """
    lib = _lib.load()
    n, h, w, cs = x.shape
    a = ConvArgs()
    a.in_ = ptr(x)
    a.n, a.h, a.w, a.cin, a.in_cs = n, h, w, (cin if cin is not None else cs), cs
    a.wpacked = ptr(wpacked)
    a.cout_pad = wpacked.shape[0]
    a.n_tile, a.kh, a.kw = n_tile, kh, kw
    a.y_off0 = -(kh // 2) if y_off0 is None else y_off0
    a.x_off0 = -(kw // 2) if x_off0 is None else x_off0
    a.bias = ptr(bias)
    if mid is not None:
        a.mid_scale, a.mid_shift = ptr(mid[0]), ptr(mid[1])
    if pre is not None:
        a.pre_scale, a.pre_shift, a.out_pre = ptr(pre[0]), ptr(pre[1]), ptr(pre[2])
        a.pre_cs, a.pre_co = pre[2].shape[-1], pre[3]
    if res1 is not None:
        a.res1, a.res1_cs, a.res1_co = ptr(res1[0]), res1[0].shape[-1], res1[1]
    if res2 is not None:
        a.res2, a.res2_cs, a.res2_co = ptr(res2[0]), res2[0].shape[-1], res2[1]
    if out_raw is not None:
        a.out_raw, a.raw_cs, a.raw_co = ptr(out_raw[0]), out_raw[0].shape[-1], out_raw[1]
    if post is not None:
        a.post_scale, a.post_shift, a.out_post = ptr(post[0]), ptr(post[1]), ptr(post[2])
        a.post_cs, a.post_co = post[2].shape[-1], post[3]
    a.out_f32 = ptr(out_f32)
    a.argmax_keys = ptr(argmax_keys)
    a.cout_real = cout_real if cout_real is not None else wpacked.shape[0]
    a.up_sy, a.up_sx, a.up_py, a.up_px = up
    a.pool2 = 1 if pool2 else 0
    if res_up is not None:
        a.res_up, a.up_cs, a.up_co = ptr(res_up[0]), res_up[0].shape[-1], res_up[1]
    check(lib.mvlm_conv2d_bf16(C.byref(a), cur_stream()), "mvlm_conv2d_bf16")


# --------------------------------------------------------------------------------------------
# stage wrappers (device tensors in, device tensors out)
# --------------------------------------------------------------------------------------------
CHANNEL_MODES = {"RGB+depth": 0, "geometry+depth": 1, "RGB": 2, "depth": 3, "geometry": 4}
MODE_CHANNELS = {0: 4, 1: 2, 2: 3, 3: 1, 4: 1}


def raster_workspace(n_views: int, h: int, w: int, n_verts: int, device) -> torch.Tensor:
    """Scratch of the rasteriser: packed depth|triangle-id keys of all pixels + per-(view, vertex) window coordinates."""
    n = _lib.load().mvlm_raster_workspace_bytes(n_views, h, w, n_verts)
    return torch.empty(((n + 7) // 8,), dtype=torch.int64, device=device)


def raster_multiview(verts, uvs, tris, tex, rot, h: int, w: int, channel_mode: str = "RGB+depth",
                     want_f32: bool = False, want_tri: bool = False, want_z: bool = False, zbuf=None, out_u8=None):
    """verts (Nv,3) f32, uvs (Nv,2) f32|None, tris (Nt,3) i32, tex (Th,Tw,3|4) u8|None, rot (V,9|3,3) f64 -- all cuda.
    zbuf: optional persistent workspace from raster_workspace().
    Returns dict(u8=(V,H,W,4) u8, f32=(V,H,W,C)|None, tri=(V,H,W) i32|None, z=(V,H,W) f32|None)."""
    lib = _lib.load()
    dev = verts.device
    mode = CHANNEL_MODES[channel_mode]
    v = rot.shape[0]
    need = lib.mvlm_raster_workspace_bytes(v, h, w, verts.shape[0])
    if zbuf is None or zbuf.numel() * zbuf.element_size() < need:
        zbuf = raster_workspace(v, h, w, verts.shape[0], dev)
    if out_u8 is None:
        out_u8 = torch.empty((v, h, w, 4), dtype=torch.uint8, device=dev)
    f32 = torch.empty((v, h, w, MODE_CHANNELS[mode]), dtype=torch.float32, device=dev) if want_f32 else None
    tri = torch.empty((v, h, w), dtype=torch.int32, device=dev) if want_tri else None
    z = torch.empty((v, h, w), dtype=torch.float32, device=dev) if want_z else None
    th, tw, tc = (tex.shape[0], tex.shape[1], tex.shape[2]) if tex is not None else (0, 0, 3)
    check(lib.mvlm_raster_multiview(ptr(verts), verts.shape[0], ptr(uvs), ptr(tris), tris.shape[0], ptr(tex), th, tw, tc,
                                    ptr(rot), v, h, w, mode, ptr(zbuf), zbuf.numel() * zbuf.element_size(), ptr(out_u8),
                                    ptr(f32), ptr(tri), ptr(z), cur_stream()),
          "mvlm_raster_multiview")
    return {"u8": out_u8, "f32": f32, "tri": tri, "z": z}


class RasterInput(NamedTuple):
    """One scan of raster_multiscan, cuda tensors as in raster_multiview.  colors: (Nv,4) u8 RGBA per-vertex colours,
    used in the RGB modes by a scan without a texture.  pages: the int32 (Nt + 3P,) table of
    mvlm_raster_multiscan_paged (the page of every triangle, then texel offset, height and width of every page), with
    tex the RGBA texels of all P pages.  render3d.DeviceMesh.raster_input builds it from a scan."""
    verts: torch.Tensor
    uvs: torch.Tensor | None
    tris: torch.Tensor
    tex: torch.Tensor | None
    colors: torch.Tensor | None = None
    pages: torch.Tensor | None = None


def raster_multiscan(scans, rot, h: int, w: int, channel_mode: str = "RGB+depth", want_f32: bool = False,
                     want_tri: bool = False, want_z: bool = False, zbuf=None, out_u8=None):
    """Several scans in one pass.  scans: list of RasterInput, or of tuples of its fields in order;
    rot (S*V,9|3,3) f64, scan-major (scan s owns views [s*V, (s+1)*V)).  zbuf: optional persistent workspace (a new
    one is allocated when it is smaller than mvlm_raster_multiscan_workspace_bytes).
    Returns dict(u8=(S*V,H,W,4), f32, tri, z) like raster_multiview; each scan's views equal raster_multiview's."""
    lib = _lib.load()
    n = len(scans)
    if not 1 <= n <= _lib.MAX_SCANS:
        raise ValueError(f"1 to {_lib.MAX_SCANS} scans per pass (got {n})")
    total = rot.shape[0]
    if total % n:
        raise ValueError(f"{total} views do not split evenly over {n} scans")
    v = total // n
    dev = scans[0][0].device
    mode = CHANNEL_MODES[channel_mode]
    table = (_lib.RasterScan * n)()
    rgba = (C.c_void_p * n)()
    paged = (C.c_void_p * n)()
    for i, (e, scan) in enumerate(zip(table, scans)):
        try:
            s = RasterInput(*scan)
        except TypeError:
            raise ValueError("a scan is (verts, uvs, tris, tex[, colors[, pages]])") from None
        if s.colors is not None and (s.colors.dtype != torch.uint8 or tuple(s.colors.shape) != (s.verts.shape[0], 4)):
            raise ValueError(f"vertex colours must be ({s.verts.shape[0]}, 4) uint8 RGBA")
        if s.pages is not None and (s.pages.dtype != torch.int32 or s.pages.dim() != 1
                                    or s.pages.numel() < s.tris.shape[0] or (s.pages.numel() - s.tris.shape[0]) % 3
                                    or s.tex is None or s.tex.shape[-1] != 4):
            raise ValueError("pages must be an int32 (Nt + 3P,) table with an RGBA texel buffer as tex")
        e.verts, e.n_verts, e.uvs = ptr(s.verts), s.verts.shape[0], ptr(s.uvs)
        e.tris, e.n_tris = ptr(s.tris), s.tris.shape[0]
        e.tex, (e.tex_h, e.tex_w, e.tex_channels) = ptr(s.tex), (s.tex.shape[:3] if s.tex is not None else (0, 0, 3))
        rgba[i], paged[i] = ptr(s.colors), ptr(s.pages)
    need = lib.mvlm_raster_multiscan_workspace_bytes(n, v, h, w, max(s[0].shape[0] for s in scans))
    if zbuf is None or zbuf.numel() * zbuf.element_size() < need:
        zbuf = torch.empty(((need + 7) // 8,), dtype=torch.int64, device=dev)
    if out_u8 is None:
        out_u8 = torch.empty((total, h, w, 4), dtype=torch.uint8, device=dev)
    f32 = torch.empty((total, h, w, MODE_CHANNELS[mode]), dtype=torch.float32, device=dev) if want_f32 else None
    tri = torch.empty((total, h, w), dtype=torch.int32, device=dev) if want_tri else None
    z = torch.empty((total, h, w), dtype=torch.float32, device=dev) if want_z else None
    check(lib.mvlm_raster_multiscan_paged(table, rgba, paged, n, ptr(rot), v, h, w, mode, ptr(zbuf),
                                          zbuf.numel() * zbuf.element_size(), ptr(out_u8), ptr(f32), ptr(tri), ptr(z),
                                          cur_stream()), "mvlm_raster_multiscan_paged")
    return {"u8": out_u8, "f32": f32, "tri": tri, "z": z}


def _on_device(device):
    device = torch.device(device)
    return torch.cuda.device(device) if device.type == "cuda" else contextlib.nullcontext()


@contextlib.contextmanager
def _plan_env(**kv):
    """Plan-build switches of the library are environment variables read by mvlm_hourglass_workspace_bytes / _create."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update(kv)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


class Hourglass:
    """Owns the device copy of a state_dict, the workspace and the planned network for a fixed
    (n_views, H, W).  `forward` runs the whole CNN (+ fused arg-max) on the current stream."""

    def __init__(self, state_dict: dict, n_landmarks: int, cin: int, n_views: int, h: int, w: int, device="cuda",
                 keep_probes: bool = False):
        """keep_probes: the intermediate tensors `probe()` returns keep their memory for the whole plan (layer-wise
        parity tests); otherwise the workspace packing reuses it (4.4 GB instead of 8 GB at 100 views of 256^2)."""
        lib = _lib.load()
        self.n_landmarks, self.cin, self.n_views, self.h, self.w = n_landmarks, cin, n_views, h, w
        self.device = torch.device(device)
        self.keep_probes = bool(keep_probes)
        # the plan's cudaMalloc / weight repacking launches and every later forward run on self.device, whatever the
        # caller's current device is
        with _on_device(self.device), _plan_env(MVLM_HG_KEEP_PROBES="1" if keep_probes else "0"):
            self._create(lib, state_dict, n_landmarks, cin, n_views, h, w)

    def _create(self, lib, state_dict, n_landmarks, cin, n_views, h, w):
        self._sd = {k: v.detach().to(self.device, torch.float32).contiguous() for k, v in state_dict.items()
                    if v.is_floating_point()}
        nbytes = lib.mvlm_hourglass_workspace_bytes(n_landmarks, cin, n_views, h, w)
        if nbytes == 0:
            raise _lib.MvlmError("mvlm_hourglass_workspace_bytes: " + lib.mvlm_last_error().decode())
        self.workspace = torch.empty((nbytes,), dtype=torch.uint8, device=self.device)
        names = list(self._sd.keys())
        arr_n = (C.c_char_p * len(names))(*[n.encode() for n in names])
        arr_p = (C.c_void_p * len(names))(*[self._sd[n].data_ptr() for n in names])
        arr_k = (C.c_longlong * len(names))(*[self._sd[n].numel() for n in names])
        handle = C.c_void_p()
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()  # the library repacks the weights on a stream of its own
        check(lib.mvlm_hourglass_create(arr_n, arr_p, arr_k, len(names), n_landmarks, cin, n_views, h, w,
                                        self.workspace.data_ptr(), nbytes, C.byref(handle)), "mvlm_hourglass_create")
        self._h = handle
        self.flops_per_view = lib.mvlm_hourglass_flops_per_view(n_landmarks, cin, h, w)
        self.num_launches = lib.mvlm_hourglass_num_launches(handle)

    def forward(self, img, want_heatmaps: bool = False, want_peaks: bool = True, graph: bool = False,
                selection_method: str = "simple"):
        """selection_method: "simple" (fused arg-max) or "moment" (31x31 centre of mass around it, windows re-evaluated
        from the last layer's input: no heat maps in memory for either)."""
        with _on_device(self.device):
            check(_lib.load().mvlm_hourglass_set_selection_method(self._h, {"simple": 0, "moment": 1}[selection_method]),
                  "mvlm_hourglass_set_selection_method")
            return self._forward(img, want_heatmaps, want_peaks, graph)

    def _forward(self, img, want_heatmaps: bool = False, want_peaks: bool = True, graph: bool = False):
        """img: (V,H,W,4) uint8 (rasteriser output) or (V,H,W,cin) float32; returns (peaks (L,V,3) f32, heatmaps|None).
        graph=True replays a CUDA graph of the launch sequence; the returned peaks tensor is then a persistent
        buffer owned by this object (overwritten by the next call)."""
        lib = _lib.load()
        assert img.shape[0] == self.n_views and img.shape[1] == self.h and img.shape[2] == self.w
        u8 = img if img.dtype == torch.uint8 else None
        f32 = img.contiguous() if img.dtype == torch.float32 else None
        if u8 is None and f32 is None:
            raise TypeError("img must be uint8 (V,H,W,4) or float32 (V,H,W,cin)")
        if f32 is not None and f32.shape[3] != self.cin:
            raise ValueError(f"expected {self.cin} channels, got {f32.shape[3]}")
        if graph and want_peaks and not want_heatmaps:
            if getattr(self, "_peaks_buf", None) is None:
                self._peaks_buf = torch.empty((self.n_landmarks, self.n_views, 3), dtype=torch.float32, device=self.device)
            check(lib.mvlm_hourglass_forward_graph(self._h, ptr(u8), ptr(f32), None, ptr(self._peaks_buf), cur_stream()),
                  "mvlm_hourglass_forward_graph")
            return self._peaks_buf, None
        peaks = torch.empty((self.n_landmarks, self.n_views, 3), dtype=torch.float32, device=self.device) if want_peaks else None
        hm = torch.empty((self.n_views, self.n_landmarks, self.h, self.w), dtype=torch.float32, device=self.device) \
            if want_heatmaps else None
        check(lib.mvlm_hourglass_forward(self._h, ptr(u8), ptr(f32), ptr(hm), ptr(peaks), cur_stream()),
              "mvlm_hourglass_forward")
        return peaks, hm

    def forward_keys(self, img, out_keys: torch.Tensor) -> None:
        """The network with its fused arg-max writing the u64 keys of this block of views into `out_keys`
        ((n_views, n_landmarks) int64, e.g. this rank's slot of an all-gather buffer); no peak kernel, CUDA-graph replay."""
        lib = _lib.load()
        assert img.shape[0] == self.n_views and img.shape[1] == self.h and img.shape[2] == self.w
        assert out_keys.dtype == torch.int64 and out_keys.is_contiguous() and out_keys.numel() == self.n_views * self.n_landmarks
        u8 = img if img.dtype == torch.uint8 else None
        f32 = img.contiguous() if img.dtype == torch.float32 else None
        with _on_device(self.device):
            check(lib.mvlm_hourglass_forward_keys(self._h, ptr(u8), ptr(f32), ptr(out_keys), cur_stream()),
                  "mvlm_hourglass_forward_keys")

    def probe(self, name: str) -> torch.Tensor:
        """Copy of an intermediate NHWC bf16 tensor (layer-wise parity tests)."""
        if not self.keep_probes:
            raise _lib.MvlmError("Hourglass.probe needs keep_probes=True (the workspace packing reuses the tensor's memory)")
        lib = _lib.load()
        p, h, w, c = C.c_void_p(), C.c_int(), C.c_int(), C.c_int()
        check(lib.mvlm_hourglass_probe(self._h, name.encode(), C.byref(p), C.byref(h), C.byref(w), C.byref(c)), "probe")
        off = p.value - self.workspace.data_ptr()
        n = self.n_views * h.value * w.value * c.value
        return self.workspace[off:off + 2 * n].view(torch.bfloat16).view(self.n_views, h.value, w.value, c.value).clone()

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                _lib.load().mvlm_hourglass_destroy(self._h)
                self._h = None
        except Exception:  # noqa: BLE001
            pass


def peaks_from_gathered_keys(keys: torch.Tensor, n_views: int, w: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """keys (world, slot_views, L) int64 gathered from all ranks -> peaks (L, n_views, 3) float32."""
    lib = _lib.load()
    world, slot_views, l = keys.shape
    if out is None:
        out = torch.empty((l, n_views, 3), dtype=torch.float32, device=keys.device)
    check(lib.mvlm_peaks_from_gathered_keys(ptr(keys), n_views, l, w, world, slot_views, ptr(out), cur_stream()),
          "mvlm_peaks_from_gathered_keys")
    return out


def heatmap_peaks(heatmaps: torch.Tensor, selection_method: str = "simple") -> torch.Tensor:
    lib = _lib.load()
    method = {"simple": 0, "moment": 1}[selection_method]
    v, l, h, w = heatmaps.shape
    hm = heatmaps.contiguous()
    out = torch.empty((l, v, 3), dtype=torch.float32, device=hm.device)
    check(lib.mvlm_heatmap_peaks(ptr(hm), v, l, h, w, method, ptr(out), cur_stream()), "mvlm_heatmap_peaks")
    return out


def rays_from_peaks(peaks: torch.Tensor, rot: torch.Tensor, image_size: int):
    lib = _lib.load()
    l, v = peaks.shape[:2]
    starts = torch.empty((l, v, 3), dtype=torch.float64, device=peaks.device)
    ends = torch.empty_like(starts)
    check(lib.mvlm_rays_from_peaks(ptr(peaks), ptr(rot), l, v, image_size, ptr(starts), ptr(ends), cur_stream()),
          "mvlm_rays_from_peaks")
    return starts, ends


def consensus(peaks, starts, ends, draws, mode: str = "quantile", threshold_quantile: float = 0.5,
              threshold_absolute: float = 0.5, dist_thres: float = 100.0, workspace=None):
    """Returns (landmarks (L,3) f64, errors (L,) f64, n_lines (L,) i32) on the device."""
    lib = _lib.load()
    if mode not in ("quantile", "absolute"):
        raise ValueError(f"Unknown mode for line matching in Estimator: {mode}")
    l, v = peaks.shape[:2]
    n_hyp = draws.shape[1]
    nbytes = lib.mvlm_consensus_workspace_bytes(l, v, n_hyp)
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty((nbytes,), dtype=torch.uint8, device=peaks.device)
    lm = torch.empty((l, 3), dtype=torch.float64, device=peaks.device)
    err = torch.empty((l,), dtype=torch.float64, device=peaks.device)
    nl = torch.empty((l,), dtype=torch.int32, device=peaks.device)
    check(lib.mvlm_consensus(ptr(peaks), ptr(starts), ptr(ends), l, v, 0 if mode == "quantile" else 1,
                             float(threshold_quantile), float(threshold_absolute), ptr(draws), n_hyp, float(dist_thres),
                             ptr(workspace), workspace.numel(), ptr(lm), ptr(err), ptr(nl), cur_stream()), "mvlm_consensus")
    return lm, err, nl


def consensus_multiscan(peaks, starts, ends, draws, n_scans: int, mode: str = "quantile", threshold_quantile: float = 0.5,
                        threshold_absolute: float = 0.5, dist_thres: float = 100.0, workspace=None):
    """Consensus of the S scans of one pass: peaks (L,S*V,3) f32, starts / ends (L,S*V,3) f64, draws (L,H,8) shared by
    every scan or (S,L,H,8) per scan.  Returns (landmarks (S,L,3) f64, errors (S,L) f64, n_lines (S,L) i32); scan s
    gets what consensus() returns for its views alone."""
    lib = _lib.load()
    if mode not in ("quantile", "absolute"):
        raise ValueError(f"Unknown mode for line matching in Estimator: {mode}")
    l, sv = peaks.shape[:2]
    if sv % n_scans:
        raise ValueError(f"{sv} views do not split evenly over {n_scans} scans")
    v = sv // n_scans
    per_scan = draws.dim() == 4
    if per_scan and draws.shape[0] != n_scans:
        raise ValueError(f"per-scan draws for {draws.shape[0]} scans, the pass has {n_scans}")
    n_hyp = draws.shape[-2]
    nbytes = lib.mvlm_consensus_multiscan_workspace_bytes(n_scans, l, v, n_hyp)
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty((nbytes,), dtype=torch.uint8, device=peaks.device)
    lm = torch.empty((n_scans, l, 3), dtype=torch.float64, device=peaks.device)
    err = torch.empty((n_scans, l), dtype=torch.float64, device=peaks.device)
    nl = torch.empty((n_scans, l), dtype=torch.int32, device=peaks.device)
    check(lib.mvlm_consensus_multiscan(ptr(peaks), ptr(starts), ptr(ends), n_scans, l, v, 0 if mode == "quantile" else 1,
                                       float(threshold_quantile), float(threshold_absolute), ptr(draws), int(per_scan),
                                       n_hyp, float(dist_thres), ptr(workspace), workspace.numel(), ptr(lm), ptr(err),
                                       ptr(nl), cur_stream()), "mvlm_consensus_multiscan")
    return lm, err, nl


# Above this many triangles building a uniform grid (memset + 7 small launches, 45-150 us) and querying it (20-50 us) beats
# the brute-force scan for ONE batch of 73 landmarks: measured crossover ~110k triangles, 4.9x at 2M
# (profiles/r1_snap_grid.txt).  A mesh that already has a grid uses it at any size (query alone: 3x at 100k, 20x at 2M).
SNAP_GRID_MIN_TRIS = int(os.environ.get("MVLM_SNAP_GRID_MIN_TRIS", "150000"))


class SnapGrid:
    """Spatial index for `snap_to_mesh` (the role vtkCellLocator plays in estimator3d.py:258-262): a uniform grid over
    the triangle centroids, built on the device from the device-resident mesh with no host round trip."""

    def __init__(self, verts, tris):
        lib = _lib.load()
        self.verts, self.tris, self.n_tris = verts, tris, tris.shape[0]
        self.buf = torch.empty((lib.mvlm_snap_grid_bytes(self.n_tris),), dtype=torch.uint8, device=verts.device)
        check(lib.mvlm_snap_grid_build(ptr(verts), ptr(tris), self.n_tris, ptr(self.buf), self.buf.numel(), cur_stream()),
              "mvlm_snap_grid_build")

    def query(self, landmarks, want_stats=False):
        lib = _lib.load()
        l = landmarks.shape[0]
        out = torch.empty((l, 3), dtype=torch.float64, device=self.verts.device)
        tid = torch.empty((l,), dtype=torch.int32, device=self.verts.device)
        stats = torch.empty((l, 2), dtype=torch.int32, device=self.verts.device) if want_stats else None
        ws = torch.empty((lib.mvlm_snap_grid_query_workspace_bytes(l, self.n_tris),), dtype=torch.uint8, device=self.verts.device)
        check(lib.mvlm_snap_grid_query(ptr(self.verts), ptr(self.tris), self.n_tris, ptr(self.buf), self.buf.numel(),
                                       ptr(landmarks), l, ptr(ws), ws.numel(), ptr(out), ptr(tid), ptr(stats), cur_stream()),
              "mvlm_snap_grid_query")
        return (out, tid, stats) if want_stats else (out, tid)

    def describe(self):
        """dims (3), oversize-list length, cell edge, largest binned triangle radius (synchronises)."""
        import ctypes as C
        d, e = (C.c_int32 * 4)(), (C.c_double * 2)()
        check(_lib.load().mvlm_debug_snap_grid_describe(ptr(self.buf), d, e, cur_stream()), "mvlm_debug_snap_grid_describe")
        return {"dims": tuple(d[:3]), "n_oversize": d[3], "cell_edge": e[0], "max_binned_radius": e[1]}


def snap_to_mesh(verts, tris, landmarks, workspace=None, grid=None):
    """Closest surface point per landmark.  grid: a SnapGrid of this mesh, "auto" (build one when the mesh has at least
    SNAP_GRID_MIN_TRIS triangles) or None (brute-force scan); every choice returns the same points and triangle ids."""
    if isinstance(grid, str):
        if grid != "auto":
            raise ValueError("grid must be a SnapGrid, 'auto' or None")
        grid = SnapGrid(verts, tris) if tris.shape[0] >= SNAP_GRID_MIN_TRIS else None
    if grid is not None:
        return grid.query(landmarks)
    lib = _lib.load()
    l, nt = landmarks.shape[0], tris.shape[0]
    nbytes = lib.mvlm_snap_workspace_bytes(l, nt)
    if workspace is None or workspace.numel() < nbytes:
        workspace = torch.empty((nbytes,), dtype=torch.uint8, device=verts.device)
    out = torch.empty((l, 3), dtype=torch.float64, device=verts.device)
    tid = torch.empty((l,), dtype=torch.int32, device=verts.device)
    check(lib.mvlm_snap_to_mesh(ptr(verts), ptr(tris), nt, ptr(landmarks), l, ptr(workspace), workspace.numel(), ptr(out),
                                ptr(tid), cur_stream()), "mvlm_snap_to_mesh")
    return out, tid


def snap_to_meshes(meshes, landmarks):
    """Closest surface points of the S scans of one pass: meshes = list of (verts, tris, SnapGrid|None), landmarks
    (S,L,3) f64.  Returns (points (S,L,3) f64, triangle ids (S,L) i32), equal to snap_to_mesh per scan."""
    lib = _lib.load()
    n, l = landmarks.shape[0], landmarks.shape[1]
    if n != len(meshes):
        raise ValueError(f"{len(meshes)} meshes for landmarks of {n} scans")
    if not 1 <= n <= _lib.MAX_SCANS:
        raise ValueError(f"1 to {_lib.MAX_SCANS} scans per pass (got {n})")
    table = (_lib.SnapMesh * n)()
    for e, (verts, tris, grid) in zip(table, meshes):
        e.verts, e.tris, e.n_tris = ptr(verts), ptr(tris), tris.shape[0]
        if grid is not None:
            e.grid, e.grid_bytes = ptr(grid.buf), grid.buf.numel()
    dev = landmarks.device
    ws = torch.empty((lib.mvlm_snap_to_meshes_workspace_bytes(table, n, l),), dtype=torch.uint8, device=dev)
    out = torch.empty((n, l, 3), dtype=torch.float64, device=dev)
    tid = torch.empty((n, l), dtype=torch.int32, device=dev)
    check(lib.mvlm_snap_to_meshes(table, n, ptr(landmarks), l, ptr(ws), ws.numel(), ptr(out), ptr(tid), cur_stream()),
          "mvlm_snap_to_meshes")
    return out, tid
