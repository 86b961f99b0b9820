/* mvlm_b200 -- C-ABI of the B200-native multi-view landmarking hot path.
 *
 * Every entry point replaces one stage of the reference's
 * Pipeline.predict_one_file (src/mvlm/pipeline/general_pipeline.py:67-131);
 * the stage it replaces is cited at each declaration (paths relative to the
 * reference tree).  Conventions:
 *   - plain C symbols, device pointers unless the name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *   - return 0 on success, <0 on error (MVLM_E_*); mvlm_last_error() gives the
 *     message of the last failing call on the calling thread;
 *   - no hidden device allocation in stage calls: the caller owns workspaces
 *     sized by the matching *_workspace_bytes() function.  Only the
 *     *_create() functions allocate (and *_destroy() frees).
 */
#ifndef MVLM_B200_H
#define MVLM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVLM_OK 0
#define MVLM_E_INVALID (-1)
#define MVLM_E_CUDA (-2)
#define MVLM_E_UNSUPPORTED (-3)

const char* mvlm_last_error(void);
int mvlm_version(void);
/* Number of kernels this library launched since the last reset (bench.py's gpu_launches). */
long long mvlm_launch_count(int reset);

/* ------------------------------------------------------------------------- */
/* Stage 2 building block: one convolution of the stacked-hourglass CNN.      */
/* Replaces torch.nn.Conv2d (+BatchNorm2d/ReLU/residual/cat) call sites:      */
/*   src/mvlm/prediction/paulsenpredictor.py:251-273, :385-402, :404-432      */
/* Activations NHWC bf16; weights packed by mvlm_pack_conv_weight().          */
/* ------------------------------------------------------------------------- */
typedef struct mvlm_conv_args {
  const void* in;      /* bf16 NHWC, channel stride in_cs */
  int n, h, w, cin, in_cs;
  const void* wpacked; /* bf16 [cout_pad][kw][kh][cin] */
  int cout_pad, n_tile, kh, kw, y_off0, x_off0;
  const float* bias;
  const float* pre_scale;
  const float* pre_shift;
  void* out_pre;
  int pre_cs, pre_co;
  const void* res1;
  int res1_cs, res1_co;
  const void* res2;
  int res2_cs, res2_co;
  void* out_raw;
  int raw_cs, raw_co;
  const float* post_scale;
  const float* post_shift;
  void* out_post;
  int post_cs, post_co;
  float* out_f32;                  /* NCHW fp32 (n, cout_real, h*up_sy, w*up_sx) */
  unsigned long long* argmax_keys; /* [n*cout_real], see mvlm_peaks_from_keys */
  int cout_real;
  int up_sy, up_sx, up_py, up_px;
  const float* mid_scale; /* optional: v = relu(v*mid_scale+mid_shift) right after the bias */
  const float* mid_shift;
  int pool2;              /* 1: out_raw / out_post are the 2x2 max-pooled (half resolution) tensors */
  const void* res_up;     /* optional bf16 (n, h/2, w/2, up_cs): v += nearest-x2 up-sampled res_up (with res1/res2) */
  int up_cs, up_co;
} mvlm_conv_args;

int mvlm_conv2d_bf16(const mvlm_conv_args* args, void* stream);

/* Debug aid: when dev_buf (mvlm_debug_conv_profile_ints() int64, device) is non-NULL the following conv launches record per-CTA role
 * stall cycles there: [0] producer wait A-empty, [1] producer wait B-empty, [2] MMA wait operands,
 * [3] MMA wait accumulator-free, [4] MMA total, [5] epilogue wait accumulator-full, [6] epilogue total,
 * [7] producer total.  NULL switches it off. */
void mvlm_debug_conv_profile(long long* dev_buf);
/* number of int64 the buffer given to mvlm_debug_conv_profile must hold (role counters + CTA-0 tile timeline) */
int mvlm_debug_conv_profile_ints(void);
/* Debug experiment switch: 1 = tensor-pipe-only timing (no TMA loads; outputs are garbage), 0 = normal. */
void mvlm_debug_conv_mode(int mode);

/* fp32 OIHW (device) -> packed bf16 [cout_pad][kw][kh][cin_pad] (device), zero padded. */
int mvlm_pack_conv_weight(const float* w_oihw, int cout, int cin, int kh, int kw, int cout_pad,
                          int cin_pad, void* out_bf16, void* stream);

/* ------------------------------------------------------------------------- */
/* Scan loader (host, multi-threaded): Wavefront OBJ -> flat arrays.            */
/* Replaces vtkOBJReader in obj_to_actor, src/mvlm/utils/utils3d.py:16-21       */
/* (error "does not contain any points" :20-21).  Output vertices are the       */
/* unique (position, vt) pairs in ascending order, faces fan-triangulated.      */
/* n_threads <= 0: one thread per host core (at most 16).                       */
/* ------------------------------------------------------------------------- */
typedef struct mvlm_obj mvlm_obj;
int mvlm_obj_load(const char* path, int n_threads, mvlm_obj** out);
int mvlm_obj_counts(const mvlm_obj* obj, int* n_verts, int* n_tris, int* has_uv);
/* verts f32[n_verts*3], uvs f32[n_verts*2] (may be NULL), tris i32[n_tris*3]: host memory */
int mvlm_obj_copy(const mvlm_obj* obj, float* verts, float* uvs, int32_t* tris);
void mvlm_obj_free(mvlm_obj* obj);
/* Materials (DESIGN.md 7g): mvlm_obj_load_ex(..., MVLM_OBJ_MATERIALS, ...) loads the same arrays as mvlm_obj_load and */
/* also keeps the `mtllib` names (rest of the line, trimmed; in file order), the distinct `usemtl` names (rest of the  */
/* line, trimmed) in order of first appearance, and each triangle's material: the index of the name of the last       */
/* `usemtl` line before its `f` line, -1 before the first.  flags = 0 is mvlm_obj_load.                                */
#define MVLM_OBJ_MATERIALS 1
int mvlm_obj_load_ex(const char* path, int n_threads, int flags, mvlm_obj** out);
/* tri_material i32[n_tris] host memory (may be NULL); an error for a scan loaded without MVLM_OBJ_MATERIALS */
int mvlm_obj_materials(const mvlm_obj* obj, int32_t* tri_material, int* n_materials, int* n_libraries);
/* NUL-terminated names owned by obj (bytes as in the file); NULL for an index out of range */
const char* mvlm_obj_material_name(const mvlm_obj* obj, int i);
const char* mvlm_obj_library_name(const mvlm_obj* obj, int i);
/* Debug (host, no file): the byte offsets where mvlm_obj_load's parallel chunks of text[0, len) start, for n_threads  */
/* as mvlm_obj_load takes it; starts holds up to 16 (or n_threads) entries; returns the number of chunks.               */
int mvlm_debug_obj_chunk_starts(const char* text, size_t len, int n_threads, long long* starts);

/* Scan loader on the GPU (obj_parse.cu): the same language, arrays and error messages as mvlm_obj_load, bit for bit, */
/* parsed from the file's bytes in device memory.  Two phases on the caller's stream:                                 */
/*   mvlm_obj_parse_device  parses up to the output sizes, synchronises `stream` and fills *info; the error of a bad   */
/*                          file (malformed line, no points, out-of-range index) is returned like mvlm_obj_load's,     */
/*                          `path` only names the file in it.  info->fallback = 1: the file holds a number of more   */
/*                          than 19 significant digits (or exceeds the parser's capacity): parse it with mvlm_obj_load */
/*   mvlm_obj_parse_write   writes verts f32[n_verts*3], uvs f32[n_verts*2] (only when has_uv), tris i32[n_tris*3]    */
/*                          into device buffers; asynchronous, reads the workspace of the first phase.                 */
/* workspace: mvlm_obj_parse_workspace_bytes(n_bytes) bytes of device memory, 256-byte aligned (0: beyond capacity). */
typedef struct mvlm_obj_parse_info {
  int32_t n_verts, n_tris, has_uv, fallback;
  int32_t n_positions; /* `v` lines */
  size_t n_bytes;
} mvlm_obj_parse_info;
size_t mvlm_obj_parse_workspace_bytes(size_t n_bytes);
int mvlm_obj_parse_device(const char* text_dev, size_t n_bytes, const char* path, void* workspace,
                          size_t workspace_bytes, void* stream, mvlm_obj_parse_info* info);
int mvlm_obj_parse_write(const mvlm_obj_parse_info* info, const void* workspace, float* verts, float* uvs,
                         int32_t* tris, void* stream);
/* Materials on the GPU (DESIGN.md 7g): mvlm_obj_parse_device_ex with MVLM_OBJ_MATERIALS parses like                    */
/* mvlm_obj_parse_device and also returns, in file order, every `usemtl` / `mtllib` line: its byte offset in the file,   */
/* its kind (1 usemtl, 2 mtllib) and the triangles of the faces before it.  The names are read by the caller from its  */
/* copy of the file (the rest of the line, trimmed, as mvlm_obj_load_ex).  name_lines: host buffer of at least          */
/* MVLM_OBJ_MAX_NAME_LINES entries; a file with more name lines sets info->fallback (mvlm_obj_load_ex reads it).        */
/* workspace: mvlm_obj_parse_workspace_bytes_ex(n_bytes, MVLM_OBJ_MATERIALS) bytes.  After mvlm_obj_parse_write,        */
/* mvlm_obj_parse_tri_page copies line_page (host, the page of every `usemtl` ordinal in file order) into the workspace */
/* and writes tri_page i32[n_tris] (device): line_page[ordinal of the last `usemtl` before the triangle], -1 before the */
/* first.  flags = 0 is mvlm_obj_parse_device / mvlm_obj_parse_workspace_bytes.                                         */
#define MVLM_OBJ_MAX_NAME_LINES 65536
typedef struct mvlm_obj_name_line {
  int64_t offset;       /* byte offset of the line's first character */
  int32_t kind;         /* 1 usemtl, 2 mtllib */
  int32_t tris_before;  /* triangles of the faces before the line */
} mvlm_obj_name_line;
size_t mvlm_obj_parse_workspace_bytes_ex(size_t n_bytes, int flags);
int mvlm_obj_parse_device_ex(const char* text_dev, size_t n_bytes, const char* path, void* workspace,
                             size_t workspace_bytes, int flags, void* stream, mvlm_obj_parse_info* info,
                             mvlm_obj_name_line* name_lines, int max_name_lines, int* n_name_lines);
int mvlm_obj_parse_tri_page(const mvlm_obj_parse_info* info, void* workspace, const int32_t* line_page, int n_usemtl,
                            int32_t* tri_page, void* stream);
/* Debug (host memory, no GPU): the GPU parser's per-line code run serially over text[0, len).  Per line: kind (0 other, */
/* 1 v, 2 vt, 3 f), status (0 ok, 1 malformed, 2 host fallback), values f32[3] (v: x y z, vt: u v), n_tris (f), and   */
/* for f lines the raw (a, b) of each triangulated corner appended to corners i64[2*max_corners] (b = 0: no uv).      */
int mvlm_debug_obj_parse_lines(const char* text, size_t len, int max_lines, int* n_lines, int32_t* kind,
                               int32_t* status, float* values, int32_t* n_tris, long long* corners,
                               long long max_corners);

/* ------------------------------------------------------------------------- */
/* Scan loader (host): PLY (ascii / binary little / big endian) and STL       */
/* (ascii / binary) -> flat arrays; the format is chosen by the suffix (.ply,  */
/* .stl, any case).  The legacy Deep-MVLM Utils3D read these formats too.      */
/* Rules (DESIGN.md 7f): PLY `vertex` x y z as float32, red green blue as      */
/* colours when all three are uchar, `face` vertex_indices fan-triangulated;   */
/* STL is binary iff its size is 84 + 50 n, and its corners are welded: equal  */
/* float32 coordinates (+0 == -0, NaN never) give one vertex, numbered in      */
/* order of first occurrence; facets made degenerate by the weld are dropped.  */
/* Errors as mvlm_obj_load ("does not exist", "does not contain any points",  */
/* "face references vertex i of n") plus malformed header / body messages.     */
/* n_threads <= 0: one thread per host core (at most 16; ASCII bodies only).   */
/* ------------------------------------------------------------------------- */
typedef struct mvlm_mesh mvlm_mesh;
int mvlm_mesh_load(const char* path, int n_threads, mvlm_mesh** out);
int mvlm_mesh_counts(const mvlm_mesh* mesh, int* n_verts, int* n_tris, int* has_colors);
/* verts f32[n_verts*3], colors u8[n_verts*3] (may be NULL), tris i32[n_tris*3]: host memory */
int mvlm_mesh_copy(const mvlm_mesh* mesh, float* verts, uint8_t* colors, int32_t* tris);
void mvlm_mesh_free(mvlm_mesh* mesh);

/* PLY / STL decoder on the GPU (mesh_parse.cu): the arrays of mvlm_mesh_load, bit for bit, for binary PLY whose faces */
/* are all triangles and for binary STL (welded on the device).  Two phases on the caller's stream, like the OBJ      */
/* parser:                                                                                                             */
/*   mvlm_mesh_parse_device  file bytes in page-locked host memory (`host`, n_bytes): parses the PLY header or checks   */
/*                           the STL size rule on the host, copies the bytes into the workspace, decodes (and welds)  */
/*                           up to the output sizes, synchronises `stream` and fills *info.  info->fallback = 1: read */
/*                           the file with mvlm_mesh_load (ASCII, a face that is not a triangle, an index out of       */
/*                           range, any PLY the fixed-stride layout does not prove, beyond capacity); errors of the    */
/*                           header are returned like mvlm_mesh_load's                                                  */
/*   mvlm_mesh_parse_write   writes verts f32[n_verts*3], colors u8[n_verts*3] (only when has_colors), tris            */
/*                           i32[n_tris*3] into device buffers; asynchronous, reads the workspace of the first phase.  */
/* workspace: mvlm_mesh_parse_workspace_bytes(n_bytes, is_stl) bytes of device memory, 256-byte aligned (0: beyond the */
/* decoder's capacity, 5.5M STL facets = the 16.7M items of one device scan, or not a binary STL size).               */
typedef struct mvlm_mesh_parse_info {
  int32_t n_verts, n_tris, has_colors, fallback;
  int32_t is_stl;
  size_t n_bytes;
} mvlm_mesh_parse_info;
size_t mvlm_mesh_parse_workspace_bytes(size_t n_bytes, int is_stl);
int mvlm_mesh_parse_device(const uint8_t* host, size_t n_bytes, int is_stl, const char* path, void* workspace,
                           size_t workspace_bytes, void* stream, mvlm_mesh_parse_info* info);
int mvlm_mesh_parse_write(const mvlm_mesh_parse_info* info, const void* workspace, float* verts, uint8_t* colors,
                          int32_t* tris, void* stream);

/* Texture decode on the GPU (nvJPEG); replaces vtkJPEGReader in obj_to_actor, src/mvlm/utils/utils3d.py:26-36.  */
/* data/len: the compressed file in host memory; out_rgb_dev: device buffer u8[height][width][3], row 0 = top.    */
/* Thread-safe (one decoder state per calling thread); asynchronous on `stream` after the host-side parse.        */
int mvlm_jpeg_info(const uint8_t* data, size_t len, int* width, int* height);
int mvlm_jpeg_decode_rgb(const uint8_t* data, size_t len, uint8_t* out_rgb_dev, int width, int height, void* stream);

/* ------------------------------------------------------------------------- */
/* Stage 1: batched multi-view orthographic rasteriser.                       */
/* Replaces ObjVTKRenderer3D.render_3d_multi_rgb_geometry_depth               */
/*   src/mvlm/utils/render3d.py:114-177 (+ camera :53-59,:136,:150-152, depth  */
/*   encoder :73-77,:166-170, flip :177, /255 :191) and obj_to_actor's         */
/*   material src/mvlm/utils/utils3d.py:26-64.                                 */
/* rot: (V,9) float64 row-major R = Ry(ry)*Rx(rx)*Rz(rz) per view.             */
/* channel_mode: 0 RGB+depth, 1 geometry+depth, 2 RGB, 3 depth, 4 geometry.    */
/* tex: (Th,Tw,tex_channels) u8, tex_channels 3 (RGB) or 4 (RGBA, one 4-byte load  */
/* per texel).  workspace: mvlm_raster_workspace_bytes(...) bytes = the packed      */
/* depth|triangle-id keys of all pixels + the per-(view, vertex) window coordinates */
/* (each vertex is transformed once per view).  Any of the four outputs may be NULL.*/
/* ------------------------------------------------------------------------- */
size_t mvlm_raster_workspace_bytes(int n_views, int h, int w, int n_verts);
int mvlm_raster_multiview(const float* verts, int n_verts, const float* uvs, const int32_t* tris, int n_tris,
                          const uint8_t* tex, int tex_h, int tex_w, int tex_channels, const double* rot,
                          int n_views, int h, int w, int channel_mode, void* workspace, size_t workspace_bytes,
                          uint8_t* out_u8 /* (V,H,W,4) */, float* out_f32 /* (V,H,W,C) */,
                          int32_t* out_tri_id /* (V,H,W) */, float* out_depth /* (V,H,W) */,
                          void* stream);

/* Several scans in one pass (the batch drivers' small-view case: one CNN plan over all views of the pass).  Views   */
/* are scan-major: global view g = s * n_views + v, rot (S*V,9), outputs (S*V,H,W,...).  Each scan's views are      */
/* rendered exactly as mvlm_raster_multiview renders them alone.  The table is passed to the kernels by value: up   */
/* to MVLM_MAX_SCANS entries, host memory, no copy to the device.  workspace:                                       */
/* mvlm_raster_multiscan_workspace_bytes(S, V, H, W, largest n_verts of the pass); for S = 1 it equals             */
/* mvlm_raster_workspace_bytes(V, H, W, n_verts).                                                                   */
#define MVLM_MAX_SCANS 64
typedef struct mvlm_raster_scan {
  const float* verts; /* (Nv,3) */
  int n_verts;
  const float* uvs;   /* (Nv,2) or NULL */
  const int32_t* tris; /* (Nt,3) */
  int n_tris;
  const uint8_t* tex; /* (Th,Tw,tex_channels) or NULL */
  int tex_h, tex_w, tex_channels;
} mvlm_raster_scan;
size_t mvlm_raster_multiscan_workspace_bytes(int n_scans, int n_views, int h, int w, int max_verts);
int mvlm_raster_multiscan(const mvlm_raster_scan* scans /* host, n_scans entries */, int n_scans,
                          const double* rot /* (S*V,9) */, int n_views, int h, int w, int channel_mode, void* workspace,
                          size_t workspace_bytes, uint8_t* out_u8 /* (S*V,H,W,4) */, float* out_f32 /* (S*V,H,W,C) */,
                          int32_t* out_tri_id /* (S*V,H,W) */, float* out_depth /* (S*V,H,W) */, void* stream);
/* The same pass with per-vertex colours: vertex_rgba[s] = scan s's (Nv,4) u8 RGBA colours in device memory (4-byte    */
/* aligned).  The entries, or the whole array (= mvlm_raster_multiscan), may be NULL.  In the RGB modes (0, 2) a scan  */
/* with colours and no (tex, uvs) pair is shaded per pixel with the barycentrics the texture lookup uses, in fp32:    */
/* c = (l0*c0 + l1*c1) + l2*c2, q = (int)(c + 0.5f) clamped to [0,255]; a texture always wins; modes 1, 3 and 4 ignore */
/* the colours.                                                                                                          */
int mvlm_raster_multiscan_colored(const mvlm_raster_scan* scans /* host, n_scans entries */,
                                  const uint8_t* const* vertex_rgba /* host array of n_scans device pointers, or NULL */,
                                  int n_scans, const double* rot /* (S*V,9) */, int n_views, int h, int w,
                                  int channel_mode, void* workspace, size_t workspace_bytes, uint8_t* out_u8,
                                  float* out_f32, int32_t* out_tri_id, float* out_depth, void* stream);
/* The same pass with texture pages (several textures per scan, DESIGN.md 7g): pages[s] = NULL, or scan s's int32      */
/* device array of n_tris + 3 P entries: the page of every triangle (-1 = none: white), then per page (texel offset,   */
/* height, width) into the scan's tex, which then holds all P pages packed as RGBA texels (tex_channels 4; tex_h and   */
/* tex_w are unused) and needs uvs.  In the RGB modes a triangle of page p takes                                       */
/* page_p[h_p-1-(floor(v h_p) mod h_p)][floor(u w_p) mod w_p], the single-texture rule with the page's sizes; a paged   */
/* scan ignores vertex colours; modes 1, 3 and 4 ignore pages.  pages (the whole array) may be NULL                    */
/* (= mvlm_raster_multiscan_colored).  Preconditions the kernels do not check (device data): every page index is -1  */
/* or in [0, P), every page has height and width >= 1, and offset + height * width <= the texels in tex; anything else */
/* is undefined behaviour (render3d.DeviceMesh.paged builds a table that satisfies them).                             */
int mvlm_raster_multiscan_paged(const mvlm_raster_scan* scans /* host, n_scans entries */,
                                const uint8_t* const* vertex_rgba /* host array of n_scans device pointers, or NULL */,
                                const int32_t* const* pages /* host array of n_scans device pointers, or NULL */,
                                int n_scans, const double* rot /* (S*V,9) */, int n_views, int h, int w, int channel_mode,
                                void* workspace, size_t workspace_bytes, uint8_t* out_u8, float* out_f32,
                                int32_t* out_tri_id, float* out_depth, void* stream);

/* ------------------------------------------------------------------------- */
/* Stage 2: stacked-hourglass heat-map CNN (MVLMModel),                       */
/*   src/mvlm/prediction/paulsenpredictor.py:364-432 driven by                 */
/*   predict_landmarks_from_images :167-217.                                   */
/* names/ptrs: the torch state_dict (fp32 device tensors, reference key names).*/
/* forward: exactly one of img_u8 (V,H,W,4 packed u8 from the rasteriser) or    */
/* img_f32 (V,H,W,cin fp32 in [0,1], the reference's image_stack layout).       */
/* out_heatmaps (V,L,H,W) fp32 and out_peaks (L,V,3) fp32 are each optional.    */
/* ------------------------------------------------------------------------- */
typedef struct mvlm_hourglass mvlm_hourglass;
size_t mvlm_hourglass_workspace_bytes(int n_landmarks, int cin, int n_views, int h, int w);
double mvlm_hourglass_flops_per_view(int n_landmarks, int cin, int h, int w);
/* numels[i] = element count of tensor i (or NULL: unchecked).  Like load_state_dict (paulsenpredictor.py:102,108)
 * a missing key or a tensor whose size does not fit this model's layer is an error (MVLM_E_INVALID), never a
 * silent misread. */
int mvlm_hourglass_create(const char* const* names, const void* const* ptrs, const long long* numels,
                          int n_entries, int n_landmarks, int cin, int n_views, int h, int w, void* workspace,
                          size_t workspace_bytes, mvlm_hourglass** out);
int mvlm_hourglass_forward(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32,
                           float* out_heatmaps, float* out_peaks, void* stream);
/* Same result as mvlm_hourglass_forward; the 144 launches are captured into a CUDA graph per distinct
 * (img, out) pointer tuple on first use and replayed afterwards (buffers must stay valid and unchanged). */
int mvlm_hourglass_forward_graph(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32,
                                 float* out_heatmaps, float* out_peaks, void* stream);
/* Peak selection of the out_peaks of forward / forward_graph (PaulsenModel.selection_method, paulsenpredictor.py:55,
 * 112-158): 0 = "simple" (the fused arg-max), 1 = "moment" (centre of mass of the 31x31 window around it, :129-156).
 * "moment" stays on the fused path: the window's heat-map values are re-evaluated from the last layer's input by a
 * small kernel, so the (V,L,H,W) fp32 heat maps are not written to memory for it either. */
int mvlm_hourglass_set_selection_method(mvlm_hourglass* net, int method);
/* View-split hand-off (SURVEY.md 8b "mvlm_allgather_peaks", 8e): when one scan's views are split over ranks, each rank
 * runs the network on its block of views with the fused arg-max of the last convolution writing its keys
 * (u64 = ordered value << 32 | ~index, n_views x n_landmarks) STRAIGHT into this rank's slot of the all-gather buffer
 * keys[world][slot_views][n_landmarks]; the host layer issues ONE in-place NCCL all-gather on that buffer
 * (torch.distributed's communicator: mvlm_b200/sharding.py::allgather_keys) and ONE kernel turns the gathered keys of
 * ALL views into peaks (L, V, 3), mapping view v to (rank, row) by the contiguous split of sharding.split_views.
 * No padding copy, no per-rank scatter. */
int mvlm_hourglass_forward_keys(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32, uint64_t* out_keys,
                                void* stream);
int mvlm_peaks_from_gathered_keys(const uint64_t* keys, int n_views, int n_landmarks, int w, int world, int slot_views,
                                  float* out_peaks /* (L, V, 3) */, void* stream);
int mvlm_hourglass_num_launches(const mvlm_hourglass* net);
/* Debug aids: per-op mean milliseconds over `reps` passes (ms_out[num_launches], host memory; out_peaks (L,V,3)
 * device), optionally the conv kernel's per-role stall cycles (roles_out[num_launches*8] host doubles, layout of
 * mvlm_debug_conv_profile, mean over CTAs), and a one-line description of op `op`. */
int mvlm_debug_hourglass_profile(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32,
                                 float* out_peaks, int reps, float* ms_out, double* roles_out, int trace_op,
                                 long long* trace_out /* 64 x 16 int64 timeline of CTA 0 of conv op trace_op, or NULL */,
                                 void* stream);
int mvlm_debug_hourglass_describe(const mvlm_hourglass* net, int op, char* buf, int buf_len);
/* layer-wise parity probes: "r3", "hg1", "sum_temp", "x10" -> NHWC bf16 tensor in the workspace */
int mvlm_hourglass_probe(const mvlm_hourglass* net, const char* name, const void** ptr, int* h, int* w, int* c);
void mvlm_hourglass_destroy(mvlm_hourglass* net);

/* ------------------------------------------------------------------------- */
/* Stage 3: heat-map peaks.  Replaces find_heat_map_maxima /                   */
/*   find_maxima_in_batch_of_heatmaps, paulsenpredictor.py:112-165.            */
/* method 0 = "simple", 1 = "moment".  heatmaps (V,L,H,W) fp32 -> (L,V,3).     */
/* ------------------------------------------------------------------------- */
int mvlm_heatmap_peaks(const float* heatmaps, int n_views, int n_landmarks, int h, int w, int method,
                       float* out_peaks, void* stream);

/* ------------------------------------------------------------------------- */
/* Stage 4: peaks -> view rays.  Replaces Estimator3D.estimate_landmark_lines  */
/*   src/mvlm/utils/estimator3d.py:31-90.  rot as in mvlm_raster_multiview.    */
/* ------------------------------------------------------------------------- */
int mvlm_rays_from_peaks(const float* peaks /* (L,V,3) */, const double* rot /* (V,9) */, int n_landmarks,
                         int n_views, int image_size, double* out_starts, double* out_ends, void* stream);

/* ------------------------------------------------------------------------- */
/* Stage 5a: filter + RANSAC + least squares.  Replaces                        */
/*   estimate_landmarks_from_lines estimator3d.py:158-183 (filters :140-155,   */
/*   RANSAC :92-137, LSQ utils3d.py:99-124).  mode 0 = quantile, 1 = absolute. */
/* draws: (L,H,8) uint32 seeded hypothesis table, line index = draw mod n.     */
/* ------------------------------------------------------------------------- */
size_t mvlm_consensus_workspace_bytes(int n_landmarks, int n_views, int n_hyp);
int mvlm_consensus(const float* peaks, const double* starts, const double* ends, int n_landmarks,
                   int n_views, int mode, double threshold_quantile, float threshold_absolute,
                   const uint32_t* draws, int n_hyp, double dist_thres, void* workspace,
                   size_t workspace_bytes, double* out_landmarks /* (L,3) */, double* out_errors /* (L) */,
                   int32_t* out_nlines /* (L) or NULL */, void* stream);

/* Several scans of one pass in the same three launches.  peaks / starts / ends are the pass's (L,S*V,3) arrays     */
/* (scan s at views [s*V, (s+1)*V)); draws: one (L,H,8) table every scan uses (draws_per_scan = 0, the seeded      */
/* estimator) or one (S,L,H,8) table (draws_per_scan = 1, the reference RNG replay).  Outputs (S,L,3), (S,L), (S,L).*/
/* Each scan gets exactly what mvlm_consensus returns for it alone.  S = 1 is mvlm_consensus.                       */
size_t mvlm_consensus_multiscan_workspace_bytes(int n_scans, int n_landmarks, int n_views, int n_hyp);
int mvlm_consensus_multiscan(const float* peaks, const double* starts, const double* ends, int n_scans,
                             int n_landmarks, int n_views, int mode, double threshold_quantile,
                             float threshold_absolute, const uint32_t* draws, int draws_per_scan, int n_hyp,
                             double dist_thres, void* workspace, size_t workspace_bytes,
                             double* out_landmarks /* (S,L,3) */, double* out_errors /* (S,L) */,
                             int32_t* out_nlines /* (S,L) or NULL */, void* stream);

/* ------------------------------------------------------------------------- */
/* Stage 5b: snap to the mesh surface.  Replaces                               */
/*   Estimator3D.project_landmarks_to_surface estimator3d.py:252-285.          */
/* ------------------------------------------------------------------------- */
size_t mvlm_snap_workspace_bytes(int n_landmarks, int n_tris);
int mvlm_snap_to_mesh(const float* verts, const int32_t* tris, int n_tris, const double* landmarks,
                      int n_landmarks, void* workspace, size_t workspace_bytes, double* out /* (L,3) */,
                      int32_t* out_tri /* (L) or NULL */, void* stream);

/* Same stage with a spatial index, for large meshes or a mesh queried more than once (the reference     */
/* builds a vtkCellLocator inside every call, estimator3d.py:258-262).  mvlm_snap_grid_build fills `grid` */
/* (mvlm_snap_grid_bytes(n_tris) bytes of device memory, 16-byte aligned) with a uniform grid over the    */
/* triangle centroids, entirely on the device; mvlm_snap_grid_query returns exactly what                  */
/* mvlm_snap_to_mesh returns (same triangle, same point); landmarks many cells away from the surface are  */
/* handed to the full scan inside the same call.  out_stats (2L ints or NULL): point-triangle tests and   */
/* shells walked per landmark (-1 = full scan).                                                           */
size_t mvlm_snap_grid_bytes(int n_tris);
size_t mvlm_snap_grid_query_workspace_bytes(int n_landmarks, int n_tris);
int mvlm_snap_grid_build(const float* verts, const int32_t* tris, int n_tris, void* grid, size_t grid_bytes,
                         void* stream);
int mvlm_snap_grid_query(const float* verts, const int32_t* tris, int n_tris, const void* grid,
                         size_t grid_bytes, const double* landmarks, int n_landmarks, void* workspace,
                         size_t workspace_bytes, double* out /* (L,3) */, int32_t* out_tri /* (L) or NULL */,
                         int32_t* out_stats /* (L,2) or NULL */, void* stream);
/* Several scans of one pass: landmarks (S,L,3) of scan s snapped to mesh s, the same points and triangles as one  */
/* mvlm_snap_to_mesh (grid = NULL) or mvlm_snap_grid_query (grid built by mvlm_snap_grid_build) per scan.  The     */
/* brute-force scan of every scan runs in one launch pair; scans with a grid add one query launch each.  The table */
/* is host memory (up to MVLM_MAX_SCANS entries).                                                                 */
typedef struct mvlm_snap_mesh {
  const float* verts;   /* (Nv,3) */
  const int32_t* tris;  /* (Nt,3) */
  int n_tris;
  const void* grid;     /* NULL or this mesh's grid */
  size_t grid_bytes;
} mvlm_snap_mesh;
size_t mvlm_snap_to_meshes_workspace_bytes(const mvlm_snap_mesh* meshes, int n_scans, int n_landmarks);
int mvlm_snap_to_meshes(const mvlm_snap_mesh* meshes, int n_scans, const double* landmarks /* (S,L,3) */,
                        int n_landmarks, void* workspace, size_t workspace_bytes, double* out /* (S,L,3) */,
                        int32_t* out_tri /* (S,L) or NULL */, void* stream);
/* debug: grid dims[3] + oversize-list length, cell edge + largest binned triangle radius (synchronises) */
int mvlm_debug_snap_grid_describe(const void* grid, int32_t* dims_nover /* [4] */, double* edge_tau /* [2] */,
                                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MVLM_B200_H */
