// C-ABI glue (include/mvlm_b200.h): error state, launch counter, thin wrappers.
#include <stdarg.h>

#include <atomic>

#include "../../include/mvlm_b200.h"
#include "common.cuh"
#include "conv_umma.cuh"
#include "hourglass.cuh"
#include "stages.cuh"

namespace mvlm {

static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int sm_count() {
  static std::atomic<int> cached[kMaxDevices];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return kNumSMs;
  int n = cached[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSMs;
    cached[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

}  // namespace mvlm

using namespace mvlm;
static_assert(kMaxScans == MVLM_MAX_SCANS, "scan table size");

extern "C" {

const char* mvlm_last_error(void) { return g_err; }

int mvlm_version(void) { return 1; }

long long mvlm_launch_count(int reset) {
  return reset ? g_launches.exchange(0) : g_launches.load();
}

void mvlm_debug_conv_profile(long long* dev_buf) { conv_set_profile_buffer(dev_buf); }
int mvlm_debug_conv_profile_ints(void) { return kConvProfInts; }
void mvlm_debug_conv_mode(int mode) { conv_set_debug_mode(mode); }

int mvlm_conv2d_bf16(const mvlm_conv_args* a, void* stream) {
  MVLM_REQUIRE(a != nullptr, "mvlm_conv2d_bf16: null args");
  ConvShape s;
  s.in = static_cast<const __nv_bfloat16*>(a->in);
  s.n = a->n; s.h = a->h; s.w = a->w; s.cin = a->cin; s.in_cs = a->in_cs;
  s.wpacked = static_cast<const __nv_bfloat16*>(a->wpacked);
  s.cout_pad = a->cout_pad; s.n_tile = a->n_tile; s.kh = a->kh; s.kw = a->kw;
  s.y_off0 = a->y_off0; s.x_off0 = a->x_off0;
  ConvEpilogue e;
  e.bias = a->bias;
  e.mid_scale = a->mid_scale; e.mid_shift = a->mid_shift;
  e.pool2 = a->pool2 != 0;
  e.pre_scale = a->pre_scale; e.pre_shift = a->pre_shift;
  e.out_pre = static_cast<__nv_bfloat16*>(a->out_pre); e.pre_cs = a->pre_cs; e.pre_co = a->pre_co;
  e.res1 = static_cast<const __nv_bfloat16*>(a->res1); e.res1_cs = a->res1_cs; e.res1_co = a->res1_co;
  e.res2 = static_cast<const __nv_bfloat16*>(a->res2); e.res2_cs = a->res2_cs; e.res2_co = a->res2_co;
  e.res_up = static_cast<const __nv_bfloat16*>(a->res_up); e.up_cs = a->up_cs; e.up_co = a->up_co;
  e.out_raw = static_cast<__nv_bfloat16*>(a->out_raw); e.raw_cs = a->raw_cs; e.raw_co = a->raw_co;
  e.post_scale = a->post_scale; e.post_shift = a->post_shift;
  e.out_post = static_cast<__nv_bfloat16*>(a->out_post); e.post_cs = a->post_cs; e.post_co = a->post_co;
  e.out_f32 = a->out_f32; e.argmax_keys = a->argmax_keys; e.cout_real = a->cout_real;
  e.up_sy = a->up_sy > 0 ? a->up_sy : 1; e.up_sx = a->up_sx > 0 ? a->up_sx : 1;
  e.up_py = a->up_py; e.up_px = a->up_px;
  ConvParams p;
  int rc = conv_plan(s, e, &p);
  if (rc != MVLM_OK) return rc;
  return conv_launch(p, static_cast<cudaStream_t>(stream));
}

int mvlm_pack_conv_weight(const float* w_oihw, int cout, int cin, int kh, int kw, int cout_pad, int cin_pad,
                          void* out_bf16, void* stream) {
  MVLM_REQUIRE(w_oihw && out_bf16, "mvlm_pack_conv_weight: null pointer");
  MVLM_REQUIRE(cout_pad >= cout && cin_pad >= cin, "mvlm_pack_conv_weight: pads smaller than dims");
  const int rc = pack_conv_weight(w_oihw, cout, cin, kh, kw, cout_pad, cin_pad, static_cast<__nv_bfloat16*>(out_bf16),
                                  static_cast<cudaStream_t>(stream));
  count_launch();
  return rc;
}

size_t mvlm_raster_workspace_bytes(int n_views, int h, int w, int n_verts) {
  return raster_workspace_bytes(n_views, h, w, n_verts);
}

int mvlm_raster_multiview(const float* verts, int n_verts, const float* uvs, const int32_t* tris, int n_tris,
                          const uint8_t* tex, int tex_h, int tex_w, int tex_channels, const double* rot, int n_views, int h,
                          int w, int channel_mode, void* workspace, size_t workspace_bytes, uint8_t* out_u8, float* out_f32,
                          int32_t* out_tri_id, float* out_depth, void* stream) {
  const mvlm_raster_scan scan = {verts, n_verts, uvs, tris, n_tris, tex, tex_h, tex_w, tex_channels};
  return mvlm_raster_multiscan(&scan, 1, rot, n_views, h, w, channel_mode, workspace, workspace_bytes, out_u8, out_f32,
                               out_tri_id, out_depth, stream);
}

size_t mvlm_raster_multiscan_workspace_bytes(int n_scans, int n_views, int h, int w, int max_verts) {
  return raster_workspace_bytes(n_scans * n_views, h, w, max_verts);
}

int mvlm_raster_multiscan(const mvlm_raster_scan* scans, int n_scans, const double* rot, int n_views, int h, int w,
                          int channel_mode, void* workspace, size_t workspace_bytes, uint8_t* out_u8, float* out_f32,
                          int32_t* out_tri_id, float* out_depth, void* stream) {
  return mvlm_raster_multiscan_colored(scans, nullptr, n_scans, rot, n_views, h, w, channel_mode, workspace,
                                       workspace_bytes, out_u8, out_f32, out_tri_id, out_depth, stream);
}

int mvlm_raster_multiscan_colored(const mvlm_raster_scan* scans, const uint8_t* const* vertex_rgba, int n_scans,
                                  const double* rot, int n_views, int h, int w, int channel_mode, void* workspace,
                                  size_t workspace_bytes, uint8_t* out_u8, float* out_f32, int32_t* out_tri_id,
                                  float* out_depth, void* stream) {
  return mvlm_raster_multiscan_paged(scans, vertex_rgba, nullptr, n_scans, rot, n_views, h, w, channel_mode, workspace,
                                     workspace_bytes, out_u8, out_f32, out_tri_id, out_depth, stream);
}

int mvlm_raster_multiscan_paged(const mvlm_raster_scan* scans, const uint8_t* const* vertex_rgba,
                                const int32_t* const* pages, int n_scans, const double* rot, int n_views, int h, int w,
                                int channel_mode, void* workspace, size_t workspace_bytes, uint8_t* out_u8,
                                float* out_f32, int32_t* out_tri_id, float* out_depth, void* stream) {
  MVLM_REQUIRE(scans, "mvlm_raster_multiscan: null scan table");
  MVLM_REQUIRE(n_scans > 0 && n_scans <= kMaxScans, "mvlm_raster_multiscan: 1 to %d scans per pass (got %d)", kMaxScans,
               n_scans);
  RasterScan table[kMaxScans];
  for (int s = 0; s < n_scans; ++s) {
    const mvlm_raster_scan& q = scans[s];
    const uchar4* colors = vertex_rgba ? reinterpret_cast<const uchar4*>(vertex_rgba[s]) : nullptr;
    MVLM_REQUIRE((reinterpret_cast<uintptr_t>(colors) & 3) == 0, "mvlm_raster_multiscan: vertex colours of scan %d not 4-byte aligned", s);
    const int* paged = pages ? pages[s] : nullptr;
    MVLM_REQUIRE(!paged || (q.tex && q.uvs && q.tex_channels == 4 && (reinterpret_cast<uintptr_t>(q.tex) & 3) == 0),
                 "mvlm_raster_multiscan: scan %d has pages but no 4-byte aligned RGBA texel buffer and uvs", s);
    table[s] = RasterScan{q.verts, q.uvs, q.tris, q.tex, colors, paged, q.n_verts, q.n_tris, q.tex_h, q.tex_w,
                          q.tex_channels};
  }
  RasterArgs a;
  a.scans = table; a.n_scans = n_scans;
  a.rot = rot; a.n_views = n_views; a.h = h; a.w = w; a.channel_mode = channel_mode;
  a.zbuf = static_cast<unsigned long long*>(workspace); a.workspace_bytes = workspace_bytes;
  a.out_u8 = out_u8; a.out_f32 = out_f32; a.out_tri = out_tri_id; a.out_z = out_depth;
  return raster_launch(a, static_cast<cudaStream_t>(stream));
}

struct mvlm_hourglass {
  HourglassNet net;
};

size_t mvlm_hourglass_workspace_bytes(int n_landmarks, int cin, int n_views, int h, int w) {
  HourglassNet dry;
  if (dry.build(nullptr, n_landmarks, cin, n_views, h, w, nullptr, 0, true) != MVLM_OK) return 0;
  return dry.workspace_needed();
}

double mvlm_hourglass_flops_per_view(int n_landmarks, int cin, int h, int w) {
  HourglassNet dry;
  if (dry.build(nullptr, n_landmarks, cin, 1, h, w, nullptr, 0, true) != MVLM_OK) return 0.0;
  return dry.flops_per_view();
}

int mvlm_hourglass_create(const char* const* names, const void* const* ptrs, const long long* numels, int n_entries,
                          int n_landmarks, int cin, int n_views, int h, int w, void* workspace, size_t workspace_bytes,
                          mvlm_hourglass** out) {
  MVLM_REQUIRE(names && ptrs && out, "mvlm_hourglass_create: null pointer");
  StateDict sd;
  for (int i = 0; i < n_entries; ++i) {
    SdEntry e;
    e.p = static_cast<const float*>(ptrs[i]);
    e.numel = numels ? numels[i] : -1;
    sd[names[i]] = e;
  }
  mvlm_hourglass* h_ = new mvlm_hourglass();
  const int rc = h_->net.build(&sd, n_landmarks, cin, n_views, h, w, workspace, workspace_bytes, false);
  if (rc != MVLM_OK) {
    delete h_;
    return rc;
  }
  *out = h_;
  return MVLM_OK;
}

int mvlm_hourglass_forward(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32, float* out_heatmaps,
                           float* out_peaks, void* stream) {
  MVLM_REQUIRE(net, "mvlm_hourglass_forward: null handle");
  return net->net.forward(img_u8, img_f32, out_heatmaps, out_peaks, static_cast<cudaStream_t>(stream));
}

int mvlm_hourglass_forward_graph(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32,
                                 float* out_heatmaps, float* out_peaks, void* stream) {
  MVLM_REQUIRE(net, "mvlm_hourglass_forward_graph: null handle");
  return net->net.forward_graph(img_u8, img_f32, out_heatmaps, out_peaks, static_cast<cudaStream_t>(stream));
}

int mvlm_hourglass_set_selection_method(mvlm_hourglass* net, int method) {
  MVLM_REQUIRE(net, "mvlm_hourglass_set_selection_method: null handle");
  return net->net.set_selection_method(method);
}

int mvlm_hourglass_forward_keys(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32, uint64_t* out_keys,
                                void* stream) {
  MVLM_REQUIRE(net, "mvlm_hourglass_forward_keys: null handle");
  return net->net.forward_keys(img_u8, img_f32, reinterpret_cast<unsigned long long*>(out_keys),
                               static_cast<cudaStream_t>(stream));
}

int mvlm_peaks_from_gathered_keys(const uint64_t* keys, int n_views, int n_landmarks, int w, int world, int slot_views,
                                  float* out_peaks, void* stream) {
  return peaks_from_gathered_keys(reinterpret_cast<const unsigned long long*>(keys), n_views, n_landmarks, w, world,
                                  slot_views, out_peaks, static_cast<cudaStream_t>(stream));
}

int mvlm_debug_hourglass_profile(mvlm_hourglass* net, const uint8_t* img_u8, const float* img_f32, float* out_peaks,
                                 int reps, float* ms_out, double* roles_out, int trace_op, long long* trace_out,
                                 void* stream) {
  MVLM_REQUIRE(net, "mvlm_debug_hourglass_profile: null handle");
  return net->net.profile_ops(img_u8, img_f32, out_peaks, reps, ms_out, roles_out, trace_op, trace_out,
                              static_cast<cudaStream_t>(stream));
}

int mvlm_debug_hourglass_describe(const mvlm_hourglass* net, int op, char* buf, int buf_len) {
  MVLM_REQUIRE(net && buf && buf_len > 0, "mvlm_debug_hourglass_describe: null pointer");
  snprintf(buf, buf_len, "%s", net->net.describe_op(op).c_str());
  return MVLM_OK;
}

int mvlm_hourglass_num_launches(const mvlm_hourglass* net) { return net ? net->net.n_ops() : 0; }

int mvlm_hourglass_probe(const mvlm_hourglass* net, const char* name, const void** ptr, int* h, int* w, int* c) {
  MVLM_REQUIRE(net && name && ptr && h && w && c, "mvlm_hourglass_probe: null pointer");
  auto it = net->net.probes.find(name);
  MVLM_REQUIRE(it != net->net.probes.end(), "mvlm_hourglass_probe: unknown probe %s", name);
  *ptr = it->second.p; *h = it->second.h; *w = it->second.w; *c = it->second.c;
  return MVLM_OK;
}

void mvlm_hourglass_destroy(mvlm_hourglass* net) { delete net; }

int mvlm_heatmap_peaks(const float* heatmaps, int n_views, int n_landmarks, int h, int w, int method,
                       float* out_peaks, void* stream) {
  return peaks_from_heatmaps(heatmaps, n_views, n_landmarks, h, w, method, out_peaks,
                             static_cast<cudaStream_t>(stream));
}

int mvlm_rays_from_peaks(const float* peaks, const double* rot, int n_landmarks, int n_views, int image_size,
                         double* out_starts, double* out_ends, void* stream) {
  return rays_from_peaks(peaks, rot, n_landmarks, n_views, image_size, out_starts, out_ends,
                         static_cast<cudaStream_t>(stream));
}

size_t mvlm_consensus_workspace_bytes(int n_landmarks, int n_views, int n_hyp) {
  return consensus_workspace_bytes(n_landmarks, n_views, n_hyp);
}

int mvlm_consensus(const float* peaks, const double* starts, const double* ends, int n_landmarks, int n_views,
                   int mode, double threshold_quantile, float threshold_absolute, const uint32_t* draws, int n_hyp,
                   double dist_thres, void* workspace, size_t workspace_bytes, double* out_landmarks,
                   double* out_errors, int32_t* out_nlines, void* stream) {
  return mvlm_consensus_multiscan(peaks, starts, ends, 1, n_landmarks, n_views, mode, threshold_quantile,
                                  threshold_absolute, draws, 0, n_hyp, dist_thres, workspace, workspace_bytes,
                                  out_landmarks, out_errors, out_nlines, stream);
}

size_t mvlm_consensus_multiscan_workspace_bytes(int n_scans, int n_landmarks, int n_views, int n_hyp) {
  return consensus_workspace_bytes(n_landmarks, n_views, n_hyp, n_scans);
}

int mvlm_consensus_multiscan(const float* peaks, const double* starts, const double* ends, int n_scans,
                             int n_landmarks, int n_views, int mode, double threshold_quantile,
                             float threshold_absolute, const uint32_t* draws, int draws_per_scan, int n_hyp,
                             double dist_thres, void* workspace, size_t workspace_bytes, double* out_landmarks,
                             double* out_errors, int32_t* out_nlines, void* stream) {
  ConsensusArgs a;
  a.peaks = peaks; a.starts = starts; a.ends = ends; a.l = n_landmarks; a.v = n_views; a.n_scans = n_scans;
  a.mode = mode;
  a.threshold_quantile = threshold_quantile; a.threshold_absolute = threshold_absolute;
  a.draws = draws; a.n_hyp = n_hyp; a.dist_thres = dist_thres;
  a.draws_scan_stride = draws_per_scan ? static_cast<size_t>(n_landmarks) * n_hyp * 8 : 0;
  a.workspace = workspace; a.workspace_bytes = workspace_bytes;
  a.out_landmarks = out_landmarks; a.out_errors = out_errors; a.out_nlines = out_nlines;
  return consensus_launch(a, static_cast<cudaStream_t>(stream));
}

size_t mvlm_snap_workspace_bytes(int n_landmarks, int n_tris) { return snap_workspace_bytes(n_landmarks, n_tris); }

int mvlm_snap_to_mesh(const float* verts, const int32_t* tris, int n_tris, const double* landmarks, int n_landmarks,
                      void* workspace, size_t workspace_bytes, double* out, int32_t* out_tri, void* stream) {
  return snap_launch(verts, tris, n_tris, landmarks, n_landmarks, workspace, workspace_bytes, out, out_tri,
                     static_cast<cudaStream_t>(stream));
}

size_t mvlm_snap_grid_bytes(int n_tris) { return snap_grid_bytes(n_tris); }

int mvlm_snap_grid_build(const float* verts, const int32_t* tris, int n_tris, void* grid, size_t grid_bytes, void* stream) {
  return snap_grid_build(verts, tris, n_tris, grid, grid_bytes, static_cast<cudaStream_t>(stream));
}

size_t mvlm_snap_grid_query_workspace_bytes(int n_landmarks, int n_tris) {
  return snap_grid_query_workspace_bytes(n_landmarks, n_tris);
}

int mvlm_snap_grid_query(const float* verts, const int32_t* tris, int n_tris, const void* grid, size_t grid_bytes,
                         const double* landmarks, int n_landmarks, void* workspace, size_t workspace_bytes, double* out,
                         int32_t* out_tri, int32_t* out_stats, void* stream) {
  return snap_grid_query(verts, tris, n_tris, grid, grid_bytes, landmarks, n_landmarks, workspace, workspace_bytes, out,
                         out_tri, out_stats, static_cast<cudaStream_t>(stream));
}

static int snap_table(const mvlm_snap_mesh* meshes, int n_scans, SnapMesh* table, const void** grids) {
  MVLM_REQUIRE(meshes, "mvlm_snap_to_meshes: null mesh table");
  MVLM_REQUIRE(n_scans > 0 && n_scans <= kMaxScans, "mvlm_snap_to_meshes: 1 to %d scans per pass (got %d)", kMaxScans,
               n_scans);
  for (int i = 0; i < n_scans; ++i) {
    table[i] = SnapMesh{meshes[i].verts, meshes[i].tris, meshes[i].n_tris};
    grids[i] = meshes[i].grid;
    MVLM_REQUIRE(!meshes[i].grid || (meshes[i].n_tris > 0 && meshes[i].grid_bytes >= snap_grid_bytes(meshes[i].n_tris)),
                 "mvlm_snap_to_meshes: grid buffer of scan %d too small", i);
  }
  return MVLM_OK;
}

size_t mvlm_snap_to_meshes_workspace_bytes(const mvlm_snap_mesh* meshes, int n_scans, int n_landmarks) {
  SnapMesh table[kMaxScans];
  const void* grids[kMaxScans];
  if (snap_table(meshes, n_scans, table, grids) != MVLM_OK) return 0;
  return snap_meshes_workspace_bytes(table, n_scans, n_landmarks);
}

int mvlm_snap_to_meshes(const mvlm_snap_mesh* meshes, int n_scans, const double* landmarks, int n_landmarks,
                        void* workspace, size_t workspace_bytes, double* out, int32_t* out_tri, void* stream) {
  SnapMesh table[kMaxScans];
  const void* grids[kMaxScans];
  const int rc = snap_table(meshes, n_scans, table, grids);
  if (rc != MVLM_OK) return rc;
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n_scans == 1 && grids[0])  // one scan with a grid: exactly mvlm_snap_grid_query's launches
    return snap_grid_query(table[0].verts, table[0].tris, table[0].nt, grids[0], meshes[0].grid_bytes, landmarks,
                           n_landmarks, workspace, workspace_bytes, out, out_tri, nullptr, s);
  return snap_meshes_launch(table, grids, n_scans, landmarks, n_landmarks, workspace, workspace_bytes, out, out_tri, s);
}

int mvlm_debug_snap_grid_describe(const void* grid, int32_t* dims_nover, double* edge_tau, void* stream) {
  return snap_grid_describe(grid, dims_nover, edge_tau, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
