// Internal launcher declarations of the non-CNN stages (one .cu per stage).
#pragma once
#include "common.cuh"

namespace mvlm {

// ---- raster.cu ------------------------------------------------------------
// Scans of one pass: the kernels take the whole table by value (a __grid_constant__ parameter), so no host -> device
// copy of it is needed.  Views of a pass are scan-major: global view g = s * n_views + v.
constexpr int kMaxScans = 64;
struct RasterScan {
  const float* verts;          // (Nv,3)
  const float* uvs;            // (Nv,2) or null
  const int* tris;             // (Nt,3)
  const unsigned char* tex;    // (Th,Tw,tex_c) or null
  const uchar4* colors;        // (Nv) RGBA vertex colours or null; used in the RGB modes when there is no (tex, uvs)
  // texture pages or null: (Nt) page per triangle (-1 = white), then (P,3) texel offset into tex (RGBA), height, width
  const int* pages;
  int nv, nt;
  int th, tw, tex_c;           // tex_c = 3 (RGB) or 4 (RGBA: one 4-byte load per texel)
};
struct RasterArgs {
  const RasterScan* scans = nullptr;  // n_scans entries (host memory)
  int n_scans = 1;
  const double* rot = nullptr;        // (S*V,9) row-major R = Ry*Rx*Rz
  int n_views = 0, h = 0, w = 0;      // n_views per scan
  int channel_mode = 0;               // 0 RGB+depth, 1 geometry+depth, 2 RGB, 3 depth, 4 geometry
  unsigned long long* zbuf = nullptr;  // workspace of raster_workspace_bytes(): (S*V,H,W) keys, then transformed vertices
  size_t workspace_bytes = 0;
  unsigned char* out_u8 = nullptr;     // (S*V,H,W,4) packed channels (CNN stem input) or null
  float* out_f32 = nullptr;            // (S*V,H,W,C) reference-layout stack or null
  int* out_tri = nullptr;              // (S*V,H,W) or null
  float* out_z = nullptr;              // (S*V,H,W) or null
};
int raster_channels(int mode);
// total_views = S * V, n_verts = the largest vertex count of the pass
size_t raster_workspace_bytes(int total_views, int h, int w, int n_verts);
int raster_launch(const RasterArgs& a, cudaStream_t stream);

// ---- peaks.cu -------------------------------------------------------------
// heatmaps (V,L,H,W) f32 -> peaks (L,V,3) f32 = (row-1, col-0.5, value); method 0 simple, 1 moment
int peaks_from_heatmaps(const float* hm, int v, int l, int h, int w, int method, float* peaks, cudaStream_t s);
// fused path: keys[v*l] written by the conv11 epilogue -> peaks (simple method only)
int peaks_from_keys(const unsigned long long* keys, int v, int l, int h, int w, float* peaks, cudaStream_t s);
// fused path, selection_method "moment": the 31x31 window around every fused arg-max is re-evaluated from the last
// layer's input x (V, h/2, w/2, x_cs) bf16 with the four 2x2 phase kernels phase_w[2a+b] ([cout][2][2][cin]) + bias
int peaks_moment_from_keys(const unsigned long long* keys, const __nv_bfloat16* x, int x_cs, int cin,
                           const __nv_bfloat16* const* phase_w, const float* bias, int v, int l, int h, int w, float* peaks,
                           cudaStream_t s);
// view-split path: keys of all ranks gathered into `world` slots of slot_views x l keys each -> peaks (l, v, 3)
int peaks_from_gathered_keys(const unsigned long long* keys, int v, int l, int w, int world, int slot_views, float* peaks,
                             cudaStream_t s);

// ---- rays.cu --------------------------------------------------------------
int rays_from_peaks(const float* peaks, const double* rot, int l, int v, int image_size, double* starts,
                    double* ends, cudaStream_t s);

// ---- consensus.cu ---------------------------------------------------------
struct ConsensusArgs {
  const float* peaks = nullptr;    // (L,S*V,3) f32, [..,2] = heat-map value
  const double* starts = nullptr;  // (L,S*V,3)
  const double* ends = nullptr;    // (L,S*V,3)
  int l = 0, v = 0;                // v: views per scan
  int n_scans = 1;
  int mode = 0;                    // 0 quantile, 1 absolute
  double threshold_quantile = 0.5;
  float threshold_absolute = 0.5f;
  const unsigned int* draws = nullptr;  // (L,H,8) uint32 raw draws, index = draw mod n_lines; (S,L,H,8) per scan
  size_t draws_scan_stride = 0;         // 0: every scan uses the same (L,H,8) table, else L*H*8
  int n_hyp = 1;
  double dist_thres = 100.0;
  void* workspace = nullptr;
  size_t workspace_bytes = 0;
  double* out_landmarks = nullptr;  // (S,L,3)
  double* out_errors = nullptr;     // (S,L)
  int* out_nlines = nullptr;        // (S,L) lines kept by the filter (optional)
};
// Per-landmark report of the final fit (DESIGN.md 7h); every pointer (S,L,...) and required when the report is asked for.
struct ConsensusReport {
  signed char* status = nullptr;   // (S,L) 0 ransac, 1 all lines (no hypothesis accepted), 2 fewer than 3 lines
  int* n_inliers = nullptr;        // (S,L) lines of the final fit
  unsigned char* inliers = nullptr;  // (S,L,V) view v's line is one of them
  double* rms = nullptr;           // (S,L)
  double* covariance = nullptr;    // (S,L,9) row-major
};
size_t consensus_workspace_bytes(int l, int v, int n_hyp, int n_scans = 1);
// report: null runs the three consensus kernels; otherwise the report kernel runs after them (one launch more)
int consensus_launch(const ConsensusArgs& a, cudaStream_t s, const ConsensusReport* report = nullptr);

// ---- snap.cu --------------------------------------------------------------
struct SnapMesh {
  const float* verts;  // (Nv,3)
  const int* tris;     // (Nt,3)
  int nt;
};
size_t snap_workspace_bytes(int l, int nt);
int snap_launch(const float* verts, const int* tris, int nt, const double* lm, int l, void* workspace,
                size_t workspace_bytes, double* out, int* out_tri, cudaStream_t s);
// uniform grid over triangle centroids: built once per mesh on the device, exact queries (same result as snap_launch)
size_t snap_grid_bytes(int nt);
int snap_grid_build(const float* verts, const int* tris, int nt, void* grid, size_t grid_bytes, cudaStream_t s);
size_t snap_grid_query_workspace_bytes(int l, int nt);
int snap_grid_query(const float* verts, const int* tris, int nt, const void* grid, size_t grid_bytes, const double* lm,
                    int l, void* workspace, size_t workspace_bytes, double* out, int* out_tri, int* out_stats,
                    cudaStream_t s);
int snap_grid_describe(const void* grid, int* dims_nover, double* edge_tau, cudaStream_t s);
// several scans of a pass: landmarks (S,L,3) -> out (S,L,3), out_tri (S,L); grids[s] = scan s's snap grid or null
// (the brute-force scan), the same points and triangles as one snap_launch / snap_grid_query per scan
size_t snap_meshes_workspace_bytes(const SnapMesh* meshes, int n_scans, int l);
int snap_meshes_launch(const SnapMesh* meshes, const void* const* grids, int n_scans, const double* lm, int l,
                       void* workspace, size_t workspace_bytes, double* out, int* out_tri, cudaStream_t s);

// ---- eltwise.cu / stem.cu ---------------------------------------------------
// out_raw/out_act may be null; scale/shift are fp32[c] (folded BN) used only when out_act != null
int pool2_act(const __nv_bfloat16* in, int n, int h, int w, int c, __nv_bfloat16* out_raw,
              const float* scale, const float* shift, __nv_bfloat16* out_act, cudaStream_t s);
int bn_relu(const __nv_bfloat16* in, size_t npix, int c, const float* scale, const float* shift,
            __nv_bfloat16* out_act, cudaStream_t s);

// u8 (N,H,W,4) [value/255] or fp32 (N,H,W,cin) image -> bf16 (N,H,W,16): channels 0..3 = hi, 4..7 = lo, rest 0
int image_to_hilo16(const unsigned char* u8, const float* f32, int cin, size_t npix, __nv_bfloat16* out,
                    cudaStream_t s);

}  // namespace mvlm
