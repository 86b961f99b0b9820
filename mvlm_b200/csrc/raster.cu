// Batched multi-view orthographic rasteriser: all V views of one mesh -- or of the S meshes of a pass, scan-major
// (global view g = s * V + v) -- in one launch sequence.  The scans of a pass come as a table passed by value
// (__grid_constant__); each block looks up its scan from g, and the grids cover the largest scan of the pass.
//
// Replaces ObjVTKRenderer3D.render_3d_multi_rgb_geometry_depth (reference
// src/mvlm/utils/render3d.py:114-177; camera :53-59,:136,:150-152; depth byte encoder
// :73-77,:166-170; row flip :177; /255 :191) and obj_to_actor's material
// (src/mvlm/utils/utils3d.py:26-64: nearest-neighbour texture, ambient 1 / diffuse 0).
//
//   raster_xform   one thread per (view, vertex): rotate the vertex (double, like
//                  vtkTransformPolyDataFilter) and map it to the window in fp32 ONCE; the (x, y, z-buffer value)
//                  triple is kept as a float4 per (view, vertex) for the two kernels below.  (Round 1 re-did this
//                  per incident triangle and again per covered pixel: ~6x + 3x redundant fp64 work, and the
//                  triangle kernel was instruction-bound on it.)
//   raster_tris    one thread per (view, triangle): three 16-byte gathers, edge functions, and an atomicMin of
//                  the packed (depth bits << 32 | triangle id) key on every covered pixel centre.  The meshes are
//                  micro-polygon (~0.5 px/triangle at 256^2, 0.1 at config 4), so the work is triangle setup plus
//                  < 1 atomic per triangle; a per-view z-buffer is 512 KB and stays in L2.  Binning triangles into
//                  screen tiles with a shared-memory z-tile (the textbook design for LARGE triangles) costs two more
//                  passes over the (view, triangle) pairs to save less than one global atomic each: DESIGN.md 7d.
//   raster_resolve one thread per pixel: winner triangle -> barycentric uv -> nearest texel (one 4-byte load from
//                  the RGBA texture, or from the triangle's page of a scan with texture pages) or, for a scan with
//                  vertex colours and no texture, the barycentric blend of its three RGBA vertex colours; depth byte,
//                  optional geometry shade; writes the u8 NHWC4 image the CNN stem consumes and, on request, the fp32
//                  (V,H,W,C) stack / triangle-id / z maps.
//
// This file is compiled with --fmad=false: every fp32 operation rounds separately, in the same
// order as oracle/csrc/oracle_native.c (built with -ffp-contract=off), so triangle-id maps and
// depth bytes are bit-identical to the CPU oracle.
#include <algorithm>

#include "common.cuh"
#include "stages.cuh"

namespace mvlm {

namespace {

constexpr unsigned long long kBgKey = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ float edge_fn(float ax, float ay, float bx, float by, float cx, float cy) {
  const float d1 = bx - ax, d2 = cy - ay, d3 = by - ay, d4 = cx - ax;
  const float p = d1 * d2;
  const float q = d3 * d4;
  return p - q;
}

struct SV {
  float sx, sy, zb;
};

__device__ __forceinline__ SV xform_vertex(const float* __restrict__ v, const double* R, float kx, float ky) {
  const double x = v[0], y = v[1], z = v[2];
  const float xr = static_cast<float>((R[0] * x + R[1] * y) + R[2] * z);
  const float yr = static_cast<float>((R[3] * x + R[4] * y) + R[5] * z);
  const float zr = static_cast<float>((R[6] * x + R[7] * y) + R[8] * z);
  SV o;
  o.sx = (xr + 150.0f) * kx;
  o.sy = (150.0f - yr) * ky;
  o.zb = (500.0f - zr) * (1.0f / 1500.0f);
  return o;
}

__device__ __forceinline__ unsigned char blend_u8(float l0, float l1, float l2, unsigned char c0, unsigned char c1,
                                                  unsigned char c2) {
  const float c = (l0 * static_cast<float>(c0) + l1 * static_cast<float>(c1)) + l2 * static_cast<float>(c2);
  return static_cast<unsigned char>(static_cast<int>(fminf(fmaxf(c + 0.5f, 0.0f), 255.0f)));
}

struct RasterScans {
  RasterScan s[kMaxScans];
};

// (view, vertex) -> window position + z-buffer value, computed once (sv[(g - g0) * sv_stride + vertex]).  The grid's x
// extent covers the largest scan of the pass; threads past their own scan's vertex count do nothing.
__global__ void __launch_bounds__(256) raster_xform_kernel(const __grid_constant__ RasterScans scans, int n_views, int g0,
                                                           const double* __restrict__ rot, int H, int W, int sv_stride,
                                                           float4* __restrict__ sv) {
  __shared__ double R[9];
  const int g = g0 + static_cast<int>(blockIdx.y);
  const RasterScan& sc = scans.s[g / n_views];
  if (threadIdx.x < 9) R[threadIdx.x] = rot[g * 9 + threadIdx.x];
  __syncthreads();
  const float kx = static_cast<float>(static_cast<double>(W) / 300.0);
  const float ky = static_cast<float>(static_cast<double>(H) / 300.0);
  float4* out = sv + static_cast<size_t>(blockIdx.y) * sv_stride;
  const int nv = sc.nv;
  const float* __restrict__ verts = sc.verts;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += gridDim.x * blockDim.x) {
    const SV a = xform_vertex(verts + 3 * i, R, kx, ky);
    out[i] = make_float4(a.sx, a.sy, a.zb, 0.f);
  }
}

__device__ __forceinline__ SV load_sv(const float4* __restrict__ sv, int i) {
  const float4 q = __ldg(sv + i);
  SV o;
  o.sx = q.x; o.sy = q.y; o.zb = q.z;
  return o;
}

__global__ void __launch_bounds__(256) raster_tris_kernel(const __grid_constant__ RasterScans scans, int n_views, int g0,
                                                          const float4* __restrict__ sv, int sv_stride, int H, int W,
                                                          unsigned long long* __restrict__ zbuf) {
  const int g = g0 + static_cast<int>(blockIdx.y);
  const RasterScan& sc = scans.s[g / n_views];
  const float4* svv = sv + static_cast<size_t>(blockIdx.y) * sv_stride;
  unsigned long long* zb = zbuf + static_cast<size_t>(g) * H * W;
  const int nt = sc.nt;
  const int* __restrict__ tris = sc.tris;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    const int i0 = __ldg(tris + 3 * t), i1 = __ldg(tris + 3 * t + 1), i2 = __ldg(tris + 3 * t + 2);
    const SV a = load_sv(svv, i0), b = load_sv(svv, i1), c = load_sv(svv, i2);
    const float minx = fminf(a.sx, fminf(b.sx, c.sx)), maxx = fmaxf(a.sx, fmaxf(b.sx, c.sx));
    const float miny = fminf(a.sy, fminf(b.sy, c.sy)), maxy = fmaxf(a.sy, fmaxf(b.sy, c.sy));
    int x0 = static_cast<int>(ceilf(minx - 0.5f)), x1 = static_cast<int>(floorf(maxx - 0.5f));
    int y0 = static_cast<int>(ceilf(miny - 0.5f)), y1 = static_cast<int>(floorf(maxy - 0.5f));
    x0 = max(x0, 0); y0 = max(y0, 0); x1 = min(x1, W - 1); y1 = min(y1, H - 1);
    if (x0 > x1 || y0 > y1) continue;  // no pixel centre inside the bounding box: most micro-polygons end here
    const float area = edge_fn(a.sx, a.sy, b.sx, b.sy, c.sx, c.sy);
    if (area == 0.0f || area != area) continue;
    for (int py = y0; py <= y1; ++py) {
      for (int px = x0; px <= x1; ++px) {
        const float cx = static_cast<float>(px) + 0.5f, cy = static_cast<float>(py) + 0.5f;
        const float w0 = edge_fn(b.sx, b.sy, c.sx, c.sy, cx, cy);
        const float w1 = edge_fn(c.sx, c.sy, a.sx, a.sy, cx, cy);
        const float w2 = edge_fn(a.sx, a.sy, b.sx, b.sy, cx, cy);
        const bool inside = area > 0.0f ? (w0 >= 0.0f && w1 >= 0.0f && w2 >= 0.0f)
                                        : (w0 <= 0.0f && w1 <= 0.0f && w2 <= 0.0f);
        if (!inside) continue;
        const float l0 = w0 / area, l1 = w1 / area, l2 = w2 / area;
        const float z = (l0 * a.zb + l1 * b.zb) + l2 * c.zb;
        if (!(z >= 0.0f && z <= 1.0f)) continue;
        const unsigned long long key =
            (static_cast<unsigned long long>(__float_as_uint(z)) << 32) | static_cast<unsigned int>(t);
        atomicMin(zb + static_cast<size_t>(py) * W + px, key);
      }
    }
  }
}

// global views g0 .. g0 + n_chunk - 1 (sv holds the transformed vertices of exactly these views)
__global__ void __launch_bounds__(256) raster_resolve_kernel(RasterArgs g, const __grid_constant__ RasterScans scans,
                                                             const float4* __restrict__ sv, int sv_stride, int g0,
                                                             int n_chunk) {
  // grid = (pixel blocks of one view, views of the chunk): 32-bit index arithmetic (three 64-bit divisions per pixel
  // were a large part of this kernel's 275 instructions per pixel)
  const unsigned int vp = blockIdx.x * blockDim.x + threadIdx.x;  // pixel within the view
  if (vp >= static_cast<unsigned int>(g.h * g.w) || static_cast<int>(blockIdx.y) >= n_chunk) return;
  const int view = g0 + static_cast<int>(blockIdx.y);
  const RasterScan& sc = scans.s[view / g.n_views];
  const int py = static_cast<int>(vp / static_cast<unsigned int>(g.w));
  const int px = static_cast<int>(vp - static_cast<unsigned int>(py) * static_cast<unsigned int>(g.w));
  const size_t pix = static_cast<size_t>(view) * g.h * g.w + vp;
  const unsigned long long key = g.zbuf[pix];
  float r = 1.0f, gr = 1.0f, bl = 1.0f, zval = 1.0f, geo = 1.0f;
  unsigned char r8 = 255, g8 = 255, b8 = 255, geo8 = 255;
  int tid = -1;
  const int mode = g.channel_mode;
  if (key != kBgKey) {
    tid = static_cast<int>(key & 0xFFFFFFFFu);
    zval = __uint_as_float(static_cast<unsigned int>(key >> 32));
    const int i0 = __ldg(sc.tris + 3 * tid), i1 = __ldg(sc.tris + 3 * tid + 1), i2 = __ldg(sc.tris + 3 * tid + 2);
    const double* R = g.rot + view * 9;
    const bool textured = sc.tex && sc.uvs;
    if ((textured || sc.colors) && (mode == 0 || mode == 2)) {
      const float4* svv = sv + static_cast<size_t>(blockIdx.y) * sv_stride;
      const SV a = load_sv(svv, i0), b = load_sv(svv, i1), c = load_sv(svv, i2);
      const float cx = static_cast<float>(px) + 0.5f, cy = static_cast<float>(py) + 0.5f;
      const float area = edge_fn(a.sx, a.sy, b.sx, b.sy, c.sx, c.sy);
      const float l0 = edge_fn(b.sx, b.sy, c.sx, c.sy, cx, cy) / area;
      const float l1 = edge_fn(c.sx, c.sy, a.sx, a.sy, cx, cy) / area;
      const float l2 = edge_fn(a.sx, a.sy, b.sx, b.sy, cx, cy) / area;
      if (textured) {  // a texture always wins over vertex colours (pages imply a texture, mvlm_raster_multiscan_paged)
        // a single texture is page 0 at texel offset 0; a paged scan reads its triangle's page (-1: no page, white)
        const int page = sc.pages ? __ldg(sc.pages + tid) : 0;
        if (page >= 0) {
          size_t off = 0;
          int th = sc.th, tw = sc.tw;
          if (sc.pages) {
            const int* e = sc.pages + sc.nt + 3 * page;
            off = static_cast<size_t>(__ldg(e)); th = __ldg(e + 1); tw = __ldg(e + 2);
          }
          const float u = (l0 * sc.uvs[2 * i0] + l1 * sc.uvs[2 * i1]) + l2 * sc.uvs[2 * i2];
          const float v = (l0 * sc.uvs[2 * i0 + 1] + l1 * sc.uvs[2 * i1 + 1]) + l2 * sc.uvs[2 * i2 + 1];
          int tx = static_cast<int>(floorf(u * static_cast<float>(tw)));
          int ty = static_cast<int>(floorf(v * static_cast<float>(th)));
          // repeat wrap; texture coordinates inside [0, 1) (the usual case) skip the two integer divisions
          if (tx < 0 || tx >= tw) { tx %= tw; if (tx < 0) tx += tw; }
          if (ty < 0 || ty >= th) { ty %= th; if (ty < 0) ty += th; }
          const size_t ti = off + static_cast<size_t>(th - 1 - ty) * tw + tx;
          if (sc.tex_c == 4) {  // RGBA texture or pages: one 4-byte load per texel
            const uchar4 q4 = __ldg(reinterpret_cast<const uchar4*>(sc.tex) + ti);
            r8 = q4.x; g8 = q4.y; b8 = q4.z;
          } else {
            const unsigned char* texel = sc.tex + ti * 3;
            r8 = texel[0]; g8 = texel[1]; b8 = texel[2];
          }
        }
      } else {  // vertex colours (Gouraud): c = (l0*c0 + l1*c1) + l2*c2 per channel, rounded half up, clamped to [0,255]
        const uchar4 c0 = __ldg(sc.colors + i0), c1 = __ldg(sc.colors + i1), c2 = __ldg(sc.colors + i2);
        r8 = blend_u8(l0, l1, l2, c0.x, c1.x, c2.x);
        g8 = blend_u8(l0, l1, l2, c0.y, c1.y, c2.y);
        b8 = blend_u8(l0, l1, l2, c0.z, c1.z, c2.z);
      }
    }
    if (mode == 1 || mode == 4) {
      double p[3][3];
      const int idx[3] = {i0, i1, i2};
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float* v3 = sc.verts + 3 * idx[k];
#pragma unroll
        for (int rr = 0; rr < 3; ++rr)
          p[k][rr] = (R[3 * rr] * v3[0] + R[3 * rr + 1] * v3[1]) + R[3 * rr + 2] * v3[2];
      }
      const double e1x = p[1][0] - p[0][0], e1y = p[1][1] - p[0][1], e1z = p[1][2] - p[0][2];
      const double e2x = p[2][0] - p[0][0], e2y = p[2][1] - p[0][1], e2z = p[2][2] - p[0][2];
      const double nx = e1y * e2z - e1z * e2y, ny = e1z * e2x - e1x * e2z, nz = e1x * e2y - e1y * e2x;
      const double nn = sqrt((nx * nx + ny * ny) + nz * nz);
      const double s = nn > 0.0 ? fabs(nz) / nn : 0.0;
      geo8 = static_cast<unsigned char>(static_cast<int>(s * 255.0 + 0.5));

    }
  }
  const int di = static_cast<int>(-255.0f * zval);
  const unsigned char d8 = static_cast<unsigned char>(di & 0xFF);
  // the fp32 stack (reference layout, /255 as render3d.py:191) is only computed when it is asked for: four IEEE
  // divisions per pixel that the fused path (u8 image for the CNN stem) never needs
  float depth = 0.f;
  if (g.out_f32) {
    r = static_cast<float>(r8) / 255.0f; gr = static_cast<float>(g8) / 255.0f; bl = static_cast<float>(b8) / 255.0f;
    geo = static_cast<float>(geo8) / 255.0f;
    depth = static_cast<float>(d8) / 255.0f;
  }
  float o[4] = {0.f, 0.f, 0.f, 0.f};
  uchar4 q = make_uchar4(0, 0, 0, 0);
  int C = 4;
  switch (mode) {
    case 0: o[0] = r; o[1] = gr; o[2] = bl; o[3] = depth; q = make_uchar4(r8, g8, b8, d8); C = 4; break;
    case 1: o[0] = geo; o[1] = depth; q = make_uchar4(geo8, d8, 0, 0); C = 2; break;
    case 2: o[0] = r; o[1] = gr; o[2] = bl; q = make_uchar4(r8, g8, b8, 0); C = 3; break;
    case 3: o[0] = depth; q = make_uchar4(d8, 0, 0, 0); C = 1; break;
    default: o[0] = geo; q = make_uchar4(geo8, 0, 0, 0); C = 1; break;
  }
  if (g.out_u8) reinterpret_cast<uchar4*>(g.out_u8)[pix] = q;
  if (g.out_f32) {
    float* dst = g.out_f32 + pix * C;
    for (int k = 0; k < C; ++k) dst[k] = o[k];
  }
  if (g.out_tri) g.out_tri[pix] = tid;
  if (g.out_z) g.out_z[pix] = zval;
}

}  // namespace

int raster_channels(int mode) {
  switch (mode) {
    case 0: return 4;
    case 1: return 2;
    case 2: return 3;
    case 3: return 1;
    case 4: return 1;
  }
  return -1;
}

// transformed vertices are kept for at most this many bytes at a time (views are processed in chunks beyond it):
// 100 views of a 50k-vertex scan are 80 MB (one chunk), config 4 (1M vertices) runs 16 views per chunk
constexpr size_t kSvBudgetBytes = 256u << 20;

static int sv_chunk_views(int n_views, int nv) {
  const size_t per_view = static_cast<size_t>(nv) * sizeof(float4);
  const size_t fit = per_view ? kSvBudgetBytes / per_view : static_cast<size_t>(n_views);
  return static_cast<int>(std::max<size_t>(1, std::min<size_t>(static_cast<size_t>(n_views), fit)));
}

size_t raster_workspace_bytes(int n_views, int h, int w, int n_verts) {  // n_views: all views of the pass
  const size_t z = (static_cast<size_t>(n_views) * h * w * sizeof(unsigned long long) + 255) & ~static_cast<size_t>(255);
  return z + static_cast<size_t>(sv_chunk_views(n_views, n_verts)) * n_verts * sizeof(float4);
}

int raster_launch(const RasterArgs& g, cudaStream_t stream) {
  MVLM_REQUIRE(g.scans && g.rot && g.zbuf, "raster: null pointer");
  MVLM_REQUIRE(g.n_scans > 0 && g.n_scans <= kMaxScans, "raster: 1 to %d scans per pass (got %d)", kMaxScans, g.n_scans);
  MVLM_REQUIRE(g.n_views > 0 && g.h > 0 && g.w > 0, "raster: bad sizes");
  MVLM_REQUIRE(static_cast<long long>(g.n_scans) * g.n_views <= 65535, "raster: at most 65535 views per pass");
  MVLM_REQUIRE(raster_channels(g.channel_mode) > 0, "raster: unknown channel_mode %d", g.channel_mode);
  RasterScans table;
  int max_nv = 0, max_nt = 0;
  for (int s = 0; s < g.n_scans; ++s) {
    const RasterScan& sc = g.scans[s];
    MVLM_REQUIRE(sc.verts && sc.tris, "raster: null pointer (scan %d)", s);
    MVLM_REQUIRE(sc.nt > 0 && sc.nv > 0, "raster: bad sizes (scan %d)", s);
    MVLM_REQUIRE(!sc.tex || sc.tex_c == 3 || sc.tex_c == 4, "raster: texture must have 3 or 4 channels (got %d)",
                 sc.tex_c);
    table.s[s] = sc;
    max_nv = std::max(max_nv, sc.nv);
    max_nt = std::max(max_nt, sc.nt);
  }
  const int total = g.n_scans * g.n_views;
  MVLM_REQUIRE(g.workspace_bytes >= raster_workspace_bytes(total, g.h, g.w, max_nv),
               "raster: workspace too small (%zu bytes given, %zu needed)", g.workspace_bytes,
               raster_workspace_bytes(total, g.h, g.w, max_nv));
  const size_t npix = static_cast<size_t>(total) * g.h * g.w;
  const size_t zbytes = (npix * sizeof(unsigned long long) + 255) & ~static_cast<size_t>(255);
  float4* sv = reinterpret_cast<float4*>(reinterpret_cast<unsigned char*>(g.zbuf) + zbytes);
  MVLM_CHECK_CUDA(cudaMemsetAsync(g.zbuf, 0xFF, npix * sizeof(unsigned long long), stream));
  // chunks of (scan, view) pairs: every view of a chunk keeps max_nv transformed vertices
  const int chunk = sv_chunk_views(total, max_nv);
  const size_t view_pix = static_cast<size_t>(g.h) * g.w;
  for (int g0 = 0; g0 < total; g0 += chunk) {
    const int nc = std::min(chunk, total - g0);
    dim3 gx(std::min(ceil_div(max_nv, 256), 1024), nc);
    raster_xform_kernel<<<gx, 256, 0, stream>>>(table, g.n_views, g0, g.rot, g.h, g.w, max_nv, sv);
    dim3 gt(std::min(ceil_div(max_nt, 256), 1024), nc);
    raster_tris_kernel<<<gt, 256, 0, stream>>>(table, g.n_views, g0, sv, max_nv, g.h, g.w, g.zbuf);
    raster_resolve_kernel<<<dim3(static_cast<unsigned>((view_pix + 255) / 256), nc), 256, 0, stream>>>(g, table, sv, max_nv,
                                                                                                       g0, nc);
    count_launch(3);
  }
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

}  // namespace mvlm
