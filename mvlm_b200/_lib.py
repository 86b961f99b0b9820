"""ctypes binding of libmvlm_b200.so (the C-ABI in include/mvlm_b200.h).

There is deliberately no fallback: if the library is missing or a call fails the
caller gets an exception.  PyTorch is used only to own device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
# MVLM_B200_LIB: another build of the same library (A/B timing of two builds on one box, tools/ab_cnn.py)
LIB_PATH = Path(os.environ.get("MVLM_B200_LIB") or _HERE / "libmvlm_b200.so")


class MvlmError(RuntimeError):
    pass


class ConvArgs(C.Structure):
    _fields_ = [
        ("in_", C.c_void_p),
        ("n", C.c_int), ("h", C.c_int), ("w", C.c_int), ("cin", C.c_int), ("in_cs", C.c_int),
        ("wpacked", C.c_void_p),
        ("cout_pad", C.c_int), ("n_tile", C.c_int), ("kh", C.c_int), ("kw", C.c_int),
        ("y_off0", C.c_int), ("x_off0", C.c_int),
        ("bias", C.c_void_p),
        ("pre_scale", C.c_void_p), ("pre_shift", C.c_void_p), ("out_pre", C.c_void_p),
        ("pre_cs", C.c_int), ("pre_co", C.c_int),
        ("res1", C.c_void_p), ("res1_cs", C.c_int), ("res1_co", C.c_int),
        ("res2", C.c_void_p), ("res2_cs", C.c_int), ("res2_co", C.c_int),
        ("out_raw", C.c_void_p), ("raw_cs", C.c_int), ("raw_co", C.c_int),
        ("post_scale", C.c_void_p), ("post_shift", C.c_void_p), ("out_post", C.c_void_p),
        ("post_cs", C.c_int), ("post_co", C.c_int),
        ("out_f32", C.c_void_p), ("argmax_keys", C.c_void_p),
        ("cout_real", C.c_int),
        ("up_sy", C.c_int), ("up_sx", C.c_int), ("up_py", C.c_int), ("up_px", C.c_int),
        ("mid_scale", C.c_void_p), ("mid_shift", C.c_void_p),
        ("pool2", C.c_int),
        ("res_up", C.c_void_p), ("up_cs", C.c_int), ("up_co", C.c_int),
    ]


class ObjParseInfo(C.Structure):
    """mvlm_obj_parse_info: what the first phase of the GPU OBJ parser found."""
    _fields_ = [("n_verts", C.c_int32), ("n_tris", C.c_int32), ("has_uv", C.c_int32), ("fallback", C.c_int32),
                ("n_positions", C.c_int32), ("n_bytes", C.c_size_t)]


class ObjNameLine(C.Structure):
    """mvlm_obj_name_line: one `usemtl` (kind 1) / `mtllib` (kind 2) line found by the GPU OBJ parser."""
    _fields_ = [("offset", C.c_int64), ("kind", C.c_int32), ("tris_before", C.c_int32)]


class MeshParseInfo(C.Structure):
    """mvlm_mesh_parse_info: what the first phase of the GPU PLY / STL decoder found."""
    _fields_ = [("n_verts", C.c_int32), ("n_tris", C.c_int32), ("has_colors", C.c_int32), ("fallback", C.c_int32),
                ("is_stl", C.c_int32), ("n_bytes", C.c_size_t)]


class RasterScan(C.Structure):
    """mvlm_raster_scan: one scan of a multi-scan raster pass (device pointers)."""
    _fields_ = [("verts", C.c_void_p), ("n_verts", C.c_int), ("uvs", C.c_void_p), ("tris", C.c_void_p),
                ("n_tris", C.c_int), ("tex", C.c_void_p), ("tex_h", C.c_int), ("tex_w", C.c_int),
                ("tex_channels", C.c_int)]


class SnapMesh(C.Structure):
    """mvlm_snap_mesh: one mesh of a multi-scan snap (device pointers, grid optional)."""
    _fields_ = [("verts", C.c_void_p), ("tris", C.c_void_p), ("n_tris", C.c_int), ("grid", C.c_void_p),
                ("grid_bytes", C.c_size_t)]


MAX_SCANS = 64  # MVLM_MAX_SCANS
OBJ_MATERIALS = 1  # MVLM_OBJ_MATERIALS
OBJ_MAX_NAME_LINES = 65536  # MVLM_OBJ_MAX_NAME_LINES

_lib = None


def load() -> C.CDLL:
    """Loads the shared library (building nothing: see mvlm_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise MvlmError(
            f"{LIB_PATH} is missing: run `python -m mvlm_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(str(LIB_PATH))
    lib.mvlm_last_error.restype = C.c_char_p
    lib.mvlm_launch_count.restype = C.c_longlong
    lib.mvlm_launch_count.argtypes = [C.c_int]
    _lib = lib
    _declare(lib)
    return lib


def _declare(lib: C.CDLL) -> None:
    vp, i32, f32, f64, u64 = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_uint64
    sigs = {
        "mvlm_version": ([], i32),
        "mvlm_conv2d_bf16": ([C.POINTER(ConvArgs), vp], i32),
        "mvlm_pack_conv_weight": ([vp, i32, i32, i32, i32, i32, i32, vp, vp], i32),
        "mvlm_raster_workspace_bytes": ([i32, i32, i32, i32], C.c_size_t),
        "mvlm_raster_multiview": ([vp, i32, vp, vp, i32, vp, i32, i32, i32, vp, i32, i32, i32, i32, vp, C.c_size_t, vp, vp,
                                   vp, vp, vp], i32),
        "mvlm_raster_multiscan_workspace_bytes": ([i32, i32, i32, i32, i32], C.c_size_t),
        "mvlm_raster_multiscan": ([C.POINTER(RasterScan), i32, vp, i32, i32, i32, i32, vp, C.c_size_t, vp, vp, vp, vp, vp],
                                  i32),
        "mvlm_raster_multiscan_colored": ([C.POINTER(RasterScan), C.POINTER(vp), i32, vp, i32, i32, i32, i32, vp,
                                           C.c_size_t, vp, vp, vp, vp, vp], i32),
        "mvlm_raster_multiscan_paged": ([C.POINTER(RasterScan), C.POINTER(vp), C.POINTER(vp), i32, vp, i32, i32, i32,
                                         i32, vp, C.c_size_t, vp, vp, vp, vp, vp], i32),
        "mvlm_hourglass_workspace_bytes": ([i32, i32, i32, i32, i32], C.c_size_t),
        "mvlm_hourglass_flops_per_view": ([i32, i32, i32, i32], f64),
        "mvlm_hourglass_create": ([C.POINTER(C.c_char_p), C.POINTER(vp), C.POINTER(C.c_longlong), i32, i32, i32, i32,
                                   i32, i32, vp, C.c_size_t, C.POINTER(vp)], i32),
        "mvlm_hourglass_forward": ([vp, vp, vp, vp, vp, vp], i32),
        "mvlm_hourglass_forward_graph": ([vp, vp, vp, vp, vp, vp], i32),
        "mvlm_hourglass_set_selection_method": ([vp, i32], i32),
        "mvlm_hourglass_forward_keys": ([vp, vp, vp, vp, vp], i32),
        "mvlm_peaks_from_gathered_keys": ([vp, i32, i32, i32, i32, i32, vp, vp], i32),
        "mvlm_hourglass_num_launches": ([vp], i32),
        "mvlm_debug_hourglass_profile": ([vp, vp, vp, vp, i32, C.POINTER(C.c_float), C.POINTER(C.c_double), i32,
                                         C.POINTER(C.c_longlong), vp], i32),
        "mvlm_debug_conv_profile_ints": ([], i32),
        "mvlm_debug_hourglass_describe": ([vp, i32, C.c_char_p, i32], i32),
        "mvlm_hourglass_probe": ([vp, C.c_char_p, C.POINTER(vp), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)], i32),
        "mvlm_hourglass_destroy": ([vp], None),
        "mvlm_obj_load": ([C.c_char_p, i32, C.POINTER(vp)], i32),
        "mvlm_obj_counts": ([vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)], i32),
        "mvlm_obj_copy": ([vp, vp, vp, vp], i32),
        "mvlm_obj_free": ([vp], None),
        "mvlm_obj_load_ex": ([C.c_char_p, i32, i32, C.POINTER(vp)], i32),
        "mvlm_obj_materials": ([vp, vp, C.POINTER(i32), C.POINTER(i32)], i32),
        "mvlm_obj_material_name": ([vp, i32], C.c_char_p),
        "mvlm_obj_library_name": ([vp, i32], C.c_char_p),
        "mvlm_debug_obj_chunk_starts": ([C.c_char_p, C.c_size_t, i32, vp], i32),
        "mvlm_obj_parse_workspace_bytes": ([C.c_size_t], C.c_size_t),
        "mvlm_obj_parse_device": ([vp, C.c_size_t, C.c_char_p, vp, C.c_size_t, vp, C.POINTER(ObjParseInfo)], i32),
        "mvlm_obj_parse_write": ([C.POINTER(ObjParseInfo), vp, vp, vp, vp, vp], i32),
        "mvlm_obj_parse_workspace_bytes_ex": ([C.c_size_t, i32], C.c_size_t),
        "mvlm_obj_parse_device_ex": ([vp, C.c_size_t, C.c_char_p, vp, C.c_size_t, i32, vp, C.POINTER(ObjParseInfo),
                                      C.POINTER(ObjNameLine), i32, C.POINTER(i32)], i32),
        "mvlm_obj_parse_tri_page": ([C.POINTER(ObjParseInfo), vp, vp, i32, vp, vp], i32),
        "mvlm_debug_obj_parse_lines": ([C.c_char_p, C.c_size_t, i32, C.POINTER(i32), vp, vp, vp, vp, vp, C.c_longlong],
                                       i32),
        "mvlm_mesh_load": ([C.c_char_p, i32, C.POINTER(vp)], i32),
        "mvlm_mesh_counts": ([vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)], i32),
        "mvlm_mesh_copy": ([vp, vp, vp, vp], i32),
        "mvlm_mesh_free": ([vp], None),
        "mvlm_mesh_parse_workspace_bytes": ([C.c_size_t, i32], C.c_size_t),
        "mvlm_mesh_parse_device": ([vp, C.c_size_t, i32, C.c_char_p, vp, C.c_size_t, vp, C.POINTER(MeshParseInfo)], i32),
        "mvlm_mesh_parse_write": ([C.POINTER(MeshParseInfo), vp, vp, vp, vp, vp], i32),
        "mvlm_jpeg_info": ([C.c_char_p, C.c_size_t, C.POINTER(i32), C.POINTER(i32)], i32),
        "mvlm_jpeg_decode_rgb": ([C.c_char_p, C.c_size_t, vp, i32, i32, vp], i32),
        "mvlm_heatmap_peaks": ([vp, i32, i32, i32, i32, i32, vp, vp], i32),
        "mvlm_rays_from_peaks": ([vp, vp, i32, i32, i32, vp, vp, vp], i32),
        "mvlm_consensus_workspace_bytes": ([i32, i32, i32], C.c_size_t),
        "mvlm_consensus": ([vp, vp, vp, i32, i32, i32, f64, f32, vp, i32, f64, vp, C.c_size_t, vp, vp, vp, vp], i32),
        "mvlm_consensus_multiscan_workspace_bytes": ([i32, i32, i32, i32], C.c_size_t),
        "mvlm_consensus_multiscan": ([vp, vp, vp, i32, i32, i32, i32, f64, f32, vp, i32, i32, f64, vp, C.c_size_t, vp, vp,
                                      vp, vp], i32),
        "mvlm_snap_workspace_bytes": ([i32, i32], C.c_size_t),
        "mvlm_snap_to_meshes_workspace_bytes": ([C.POINTER(SnapMesh), i32, i32], C.c_size_t),
        "mvlm_snap_to_meshes": ([C.POINTER(SnapMesh), i32, vp, i32, vp, C.c_size_t, vp, vp, vp], i32),
        "mvlm_snap_to_mesh": ([vp, vp, i32, vp, i32, vp, C.c_size_t, vp, vp, vp], i32),
        "mvlm_snap_grid_bytes": ([i32], C.c_size_t),
        "mvlm_snap_grid_build": ([vp, vp, i32, vp, C.c_size_t, vp], i32),
        "mvlm_snap_grid_query_workspace_bytes": ([i32, i32], C.c_size_t),
        "mvlm_snap_grid_query": ([vp, vp, i32, vp, C.c_size_t, vp, i32, vp, C.c_size_t, vp, vp, vp, vp], i32),
        "mvlm_debug_snap_grid_describe": ([vp, vp, vp, vp], i32),
    }
    sigs.update(_EXTRA_SIGS)
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype


# filled by the per-stage binding modules below (kept in one dict so that the
# symbol-export test can iterate over everything the header declares)
_EXTRA_SIGS: dict = {}


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().mvlm_last_error().decode("utf-8", "replace")
        raise MvlmError(f"{what or 'mvlm call'} failed ({rc}): {msg}")


def ptr(t) -> int | None:
    """data_ptr of a torch tensor (or None)."""
    if t is None:
        return None
    return t.data_ptr()


def cur_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
