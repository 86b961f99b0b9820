// Snap landmarks to the closest point of the triangle mesh (exact, brute force over all triangles).
//
// Replaces Estimator3D.project_landmarks_to_surface (reference src/mvlm/utils/estimator3d.py:252-285):
// vtkCellLocator.FindClosestPoint returns the exact closest point on the mesh; the locator is only
// an accelerator, so a full scan gives the same answer.  Ties -> lowest triangle id.
// grid (L, splits): each block scans a slice of the triangles (vertex/index arrays are L2-resident:
// 1.8 MB for 100k triangles), block-reduces (dist^2, tri) and a finalize kernel picks the winner.
//
// Second path for large meshes (SURVEY.md 8f rank 3; the reference rebuilds a vtkCellLocator per call,
// estimator3d.py:258-262): a uniform grid over the triangle CENTROIDS, built on the device with no host
// round trip (bounds -> cell size -> count -> scan -> fill), and a one-warp-per-landmark query that walks
// Chebyshev shells of cells around the landmark until no unvisited triangle can beat the best one.
// Exactness: a triangle with centroid-to-vertex radius rho lies within rho of its centroid, so after all
// cells within r shells are visited every unvisited triangle is at least lb(r) - tau away (tau = largest
// binned rho; larger triangles sit in an "oversize" list every query scans).  The search stops only when
// best < lb(r) - tau STRICTLY, candidates are compared as (dist^2, triangle id) with the same arithmetic as
// the brute-force scan, so both paths return the same triangle and the same point bit for bit.
#include <cub/block/block_reduce.cuh>

#include "common.cuh"
#include "scan.cuh"
#include "stages.cuh"

namespace mvlm {

namespace {

constexpr int kSnapPart = 5;  // d2, tri, p[3]

__device__ void closest_on_tri(const double* p, const double* a, const double* b, const double* c, double* out) {
  double ab[3], ac[3], ap[3], bp[3], cp[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) { ab[i] = b[i] - a[i]; ac[i] = c[i] - a[i]; ap[i] = p[i] - a[i]; }
  const double d1 = ab[0] * ap[0] + ab[1] * ap[1] + ab[2] * ap[2];
  const double d2 = ac[0] * ap[0] + ac[1] * ap[1] + ac[2] * ap[2];
  if (d1 <= 0.0 && d2 <= 0.0) { out[0] = a[0]; out[1] = a[1]; out[2] = a[2]; return; }
#pragma unroll
  for (int i = 0; i < 3; ++i) bp[i] = p[i] - b[i];
  const double d3 = ab[0] * bp[0] + ab[1] * bp[1] + ab[2] * bp[2];
  const double d4 = ac[0] * bp[0] + ac[1] * bp[1] + ac[2] * bp[2];
  if (d3 >= 0.0 && d4 <= d3) { out[0] = b[0]; out[1] = b[1]; out[2] = b[2]; return; }
  const double vc = d1 * d4 - d3 * d2;
  if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
    const double v = d1 / (d1 - d3);
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = a[i] + v * ab[i];
    return;
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) cp[i] = p[i] - c[i];
  const double d5 = ab[0] * cp[0] + ab[1] * cp[1] + ab[2] * cp[2];
  const double d6 = ac[0] * cp[0] + ac[1] * cp[1] + ac[2] * cp[2];
  if (d6 >= 0.0 && d5 <= d6) { out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; return; }
  const double vb = d5 * d2 - d1 * d6;
  if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
    const double w = d2 / (d2 - d6);
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = a[i] + w * ac[i];
    return;
  }
  const double va = d3 * d6 - d5 * d4;
  if (va <= 0.0 && (d4 - d3) >= 0.0 && (d5 - d6) >= 0.0) {
    const double w = (d4 - d3) / ((d4 - d3) + (d5 - d6));
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = b[i] + w * (c[i] - b[i]);
    return;
  }
  const double denom = 1.0 / (va + vb + vc);
  const double v = vb * denom, w = vc * denom;
#pragma unroll
  for (int i = 0; i < 3; ++i) out[i] = a[i] + ab[i] * v + ac[i] * w;
}

__device__ __forceinline__ double tri_dist2(const float* __restrict__ verts, const int* __restrict__ tris, int t,
                                            const double* p) {
  const int i0 = __ldg(tris + 3 * t), i1 = __ldg(tris + 3 * t + 1), i2 = __ldg(tris + 3 * t + 2);
  const double a[3] = {verts[3 * i0], verts[3 * i0 + 1], verts[3 * i0 + 2]};
  const double b[3] = {verts[3 * i1], verts[3 * i1 + 1], verts[3 * i1 + 2]};
  const double c[3] = {verts[3 * i2], verts[3 * i2 + 1], verts[3 * i2 + 2]};
  double q[3];
  closest_on_tri(p, a, b, c, q);
  const double dx = q[0] - p[0], dy = q[1] - p[1], dz = q[2] - p[2];
  return dx * dx + dy * dy + dz * dz;
}

__device__ __forceinline__ void tri_closest(const float* __restrict__ verts, const int* __restrict__ tris, int t,
                                            const double* p, double* q) {
  const int i0 = tris[3 * t], i1 = tris[3 * t + 1], i2 = tris[3 * t + 2];
  const double a[3] = {verts[3 * i0], verts[3 * i0 + 1], verts[3 * i0 + 2]};
  const double b[3] = {verts[3 * i1], verts[3 * i1 + 1], verts[3 * i1 + 2]};
  const double c[3] = {verts[3 * i2], verts[3 * i2 + 1], verts[3 * i2 + 2]};
  closest_on_tri(p, a, b, c, q);
}

struct SnapMeshes {
  SnapMesh m[kMaxScans];
};

// grid (L, splits, S): landmarks lm (S,L,3) of scan s = blockIdx.z against mesh s; partial minima part (S,L,splits,5)
__global__ void __launch_bounds__(256) snap_scan_kernel(const __grid_constant__ SnapMeshes meshes, int L,
                                                        const double* __restrict__ lm, int splits,
                                                        double* __restrict__ part, const int* __restrict__ only) {
  const int l = blockIdx.z * L + blockIdx.x, split = blockIdx.y;  // (scan, landmark) slot
  if (only && !only[l]) return;  // grid path: only the landmarks its query handed back
  const SnapMesh& mesh = meshes.m[blockIdx.z];
  const float* __restrict__ verts = mesh.verts;
  const int* __restrict__ tris = mesh.tris;
  const int nt = mesh.nt;
  const double p[3] = {lm[3 * l], lm[3 * l + 1], lm[3 * l + 2]};
  const int chunk = (nt + splits - 1) / splits;
  const int t0 = split * chunk, t1 = min(nt, t0 + chunk);
  double best = INFINITY;
  int bt = 0x7fffffff;
  for (int t = t0 + threadIdx.x; t < t1; t += blockDim.x) {
    const double d = tri_dist2(verts, tris, t, p);
    if (d < best) { best = d; bt = t; }  // increasing t per thread: first minimum kept
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, best, o);
    const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
    if (od < best || (od == best && ot < bt)) { best = od; bt = ot; }
  }
  __shared__ double sd[8];
  __shared__ int st[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sd[warp] = best; st[warp] = bt; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w)
      if (sd[w] < best || (sd[w] == best && st[w] < bt)) { best = sd[w]; bt = st[w]; }
    double* o = part + (static_cast<size_t>(l) * splits + split) * kSnapPart;
    o[0] = best;
    o[1] = static_cast<double>(bt);
    if (bt != 0x7fffffff) {
      tri_closest(verts, tris, bt, p, o + 2);
    } else {
      o[2] = p[0]; o[3] = p[1]; o[4] = p[2];
    }
  }
}

// one thread per (scan, landmark) slot of the S*L
__global__ void snap_finalize_kernel(const double* __restrict__ part, int L, int splits, double* __restrict__ out,
                                     int* __restrict__ out_tri, const int* __restrict__ only) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= L || (only && !only[l])) return;
  const double* q = part + static_cast<size_t>(l) * splits * kSnapPart;
  int bs = 0;
  for (int s = 1; s < splits; ++s)
    if (q[s * kSnapPart] < q[bs * kSnapPart] ||
        (q[s * kSnapPart] == q[bs * kSnapPart] && q[s * kSnapPart + 1] < q[bs * kSnapPart + 1]))
      bs = s;
  out[3 * l] = q[bs * kSnapPart + 2];
  out[3 * l + 1] = q[bs * kSnapPart + 3];
  out[3 * l + 2] = q[bs * kSnapPart + 4];
  if (out_tri) out_tri[l] = static_cast<int>(q[bs * kSnapPart + 1]);
}

int snap_splits(int l, int nt) {
  int s = ceil_div(4 * sm_count(), l);
  const int max_s = ceil_div(nt, 256);
  if (s > max_s) s = max_s;
  return s < 1 ? 1 : s;
}

}  // namespace

// l: landmarks x scans, nt: the largest triangle count
size_t snap_workspace_bytes(int l, int nt) {
  return static_cast<size_t>(l) * snap_splits(l, nt) * kSnapPart * sizeof(double) + 64;
}

size_t snap_meshes_workspace_bytes(const SnapMesh* meshes, int n_scans, int l) {
  int max_nt = 0;
  for (int i = 0; i < n_scans; ++i) max_nt = max(max_nt, meshes[i].nt);
  const size_t part = snap_workspace_bytes(l * n_scans, max_nt);
  return part + (static_cast<size_t>(l) * n_scans * sizeof(int) + 63) / 64 * 64;
}

// The scan kernels of every scan of the pass in one launch pair.  `only` (S*L ints, device, or null): slots to do.
static int snap_scan_launch(const SnapMesh* meshes, int n_scans, const double* lm, int l, double* part, double* out,
                            int* out_tri, const int* only, cudaStream_t s) {
  SnapMeshes table;
  int max_nt = 0;
  for (int i = 0; i < n_scans; ++i) {
    table.m[i] = meshes[i];
    max_nt = max(max_nt, meshes[i].nt);
  }
  const int slots = l * n_scans;
  // splits from all slots of the pass and the largest mesh: a split of a smaller mesh may be empty; the
  // (dist^2, triangle) minimum does not depend on how the triangles are split
  const int splits = snap_splits(slots, max_nt);
  snap_scan_kernel<<<dim3(l, splits, n_scans), 256, 0, s>>>(table, l, lm, splits, part, only);
  snap_finalize_kernel<<<ceil_div(slots, 128), 128, 0, s>>>(part, slots, splits, out, out_tri, only);
  count_launch(2);
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

static int check_meshes(const SnapMesh* meshes, int n_scans) {
  MVLM_REQUIRE(meshes && n_scans > 0 && n_scans <= kMaxScans, "snap: 1 to %d scans per pass (got %d)", kMaxScans,
               n_scans);
  for (int i = 0; i < n_scans; ++i) {
    MVLM_REQUIRE(meshes[i].verts && meshes[i].tris, "snap: null pointer (scan %d)", i);
    MVLM_REQUIRE(meshes[i].nt > 0, "snap: bad sizes (scan %d)", i);
  }
  return MVLM_OK;
}

int snap_launch(const float* verts, const int* tris, int nt, const double* lm, int l, void* workspace,
                size_t workspace_bytes, double* out, int* out_tri, cudaStream_t s) {
  MVLM_REQUIRE(verts && tris && lm && out && workspace, "snap: null pointer");
  MVLM_REQUIRE(nt > 0 && l > 0, "snap: bad sizes");
  MVLM_REQUIRE(workspace_bytes >= snap_workspace_bytes(l, nt), "snap: workspace too small");
  const SnapMesh mesh = {verts, tris, nt};
  return snap_scan_launch(&mesh, 1, lm, l, static_cast<double*>(workspace), out, out_tri, nullptr, s);
}

// ---------------------------------------------------------------------------------------------------------
// Uniform-grid path
// ---------------------------------------------------------------------------------------------------------
namespace {

constexpr int kMaxShells = 8;     // shells walked before a query hands its landmark to the full scan (see 7c: a long walk
                                  // costs more than the scan, which then bounds the worst case at scan + ~50 us)
constexpr int kGridHdrBytes = 256;

struct GridHdr {
  double mn[3];
  double c, inv_c;
  double sum_rho;
  int dim[3];
  int n_over;
  unsigned int nmin_key[3], max_key[3];  // ~key(min) and key(max) so that a zero fill is the identity of atomicMax
  unsigned int tau_key;                  // key(max rho of the binned triangles), float rounded up
  int nt, cap_cells;
};
static_assert(sizeof(GridHdr) <= kGridHdrBytes, "grid header");

struct GridLayout {
  int cap_cells;
  size_t counts, cell_start, block_sums, sorted, over, total;
};

GridLayout grid_layout(int nt) {
  GridLayout g;
  long long cap = 8ll * nt;
  if (cap < kScanItems) cap = kScanItems;
  if (cap > (1ll << 24)) cap = 1ll << 24;
  g.cap_cells = static_cast<int>((cap + kScanItems - 1) / kScanItems * kScanItems);
  size_t o = kGridHdrBytes;
  g.counts = o;      o += static_cast<size_t>(g.cap_cells) * 4;
  g.cell_start = o;  o += (static_cast<size_t>(g.cap_cells) + 4) * 4;
  g.block_sums = o;  o += (static_cast<size_t>(g.cap_cells) / kScanItems + 4) * 4;
  g.sorted = o;      o += (static_cast<size_t>(nt) + 4) / 4 * 16;
  g.over = o;        o += (static_cast<size_t>(nt) + 4) / 4 * 16;
  g.total = o;
  return g;
}

__device__ __forceinline__ unsigned int float_key(float f) {
  const unsigned int u = __float_as_uint(f);
  return u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float key_float(unsigned int k) {
  return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu));
}

// centroid and centroid-to-vertex radius of triangle t (identical arithmetic in count and fill)
__device__ __forceinline__ double tri_centroid(const float* __restrict__ verts, const int* __restrict__ tris, int t,
                                               double* g) {
  const int i0 = __ldg(tris + 3 * t), i1 = __ldg(tris + 3 * t + 1), i2 = __ldg(tris + 3 * t + 2);
  double a[3], b[3], c[3], r2 = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    a[i] = verts[3 * i0 + i]; b[i] = verts[3 * i1 + i]; c[i] = verts[3 * i2 + i];
    g[i] = (a[i] + b[i] + c[i]) * (1.0 / 3.0);
  }
  double da = 0.0, db = 0.0, dc = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    da += (a[i] - g[i]) * (a[i] - g[i]); db += (b[i] - g[i]) * (b[i] - g[i]); dc += (c[i] - g[i]) * (c[i] - g[i]);
  }
  r2 = fmax(da, fmax(db, dc));
  return sqrt(r2);
}

__device__ __forceinline__ int cell_of(const GridHdr& h, const double* x) {
  int idx[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int v = static_cast<int>(floor((x[i] - h.mn[i]) * h.inv_c));
    idx[i] = min(max(v, 0), h.dim[i] - 1);
  }
  return (idx[2] * h.dim[1] + idx[1]) * h.dim[0] + idx[0];
}

__global__ void __launch_bounds__(256) grid_bounds_kernel(const float* __restrict__ verts, const int* __restrict__ tris,
                                                          int nt, GridHdr* hdr) {
  float mn[3] = {INFINITY, INFINITY, INFINITY}, mx[3] = {-INFINITY, -INFINITY, -INFINITY};
  double rho = 0.0;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    double g[3];
    rho += tri_centroid(verts, tris, t, g);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int v = __ldg(tris + 3 * t + k);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const float x = verts[3 * v + i];
        mn[i] = fminf(mn[i], x);
        mx[i] = fmaxf(mx[i], x);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      mn[i] = fminf(mn[i], __shfl_xor_sync(0xffffffffu, mn[i], o));
      mx[i] = fmaxf(mx[i], __shfl_xor_sync(0xffffffffu, mx[i], o));
    }
    rho += __shfl_xor_sync(0xffffffffu, rho, o);
  }
  if ((threadIdx.x & 31) == 0 && mn[0] <= mx[0]) {
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      atomicMax(&hdr->nmin_key[i], ~float_key(mn[i]));
      atomicMax(&hdr->max_key[i], float_key(mx[i]));
    }
    atomicAdd(&hdr->sum_rho, rho);
  }
}

// one thread: cell edge = 2.5 x the mean triangle radius, enlarged until the grid fits the cell budget
__global__ void grid_setup_kernel(GridHdr* hdr, int nt, int cap_cells) {
  double ext[3], emax = 0.0;
  for (int i = 0; i < 3; ++i) {
    const double lo = key_float(~hdr->nmin_key[i]), hi = key_float(hdr->max_key[i]);
    hdr->mn[i] = lo;
    ext[i] = hi - lo;
    if (!(ext[i] >= 0.0)) ext[i] = 0.0;  // also catches NaN
    emax = fmax(emax, ext[i]);
  }
  double c = 2.5 * hdr->sum_rho / nt;
  if (!(c > 0.0) || !(c < INFINITY)) c = emax > 0.0 ? emax : 1.0;
  int dim[3];
  for (int it = 0; it < 400; ++it) {
    double cells = 1.0;
    for (int i = 0; i < 3; ++i) {
      const double d = floor(ext[i] / c) + 1.0;
      dim[i] = d < 1024.0 ? static_cast<int>(d) : 1024;
      cells *= dim[i];
    }
    bool fits = cells <= static_cast<double>(cap_cells);
    for (int i = 0; i < 3; ++i) fits = fits && (floor(ext[i] / c) + 1.0 <= 1024.0);
    if (fits) break;
    c *= 1.1;
  }
  if (static_cast<double>(dim[0]) * dim[1] * dim[2] > cap_cells) dim[0] = dim[1] = dim[2] = 1;  // unreachable safety net
  for (int i = 0; i < 3; ++i) hdr->dim[i] = dim[i];
  hdr->c = c;
  hdr->inv_c = 1.0 / c;
  hdr->nt = nt;
  hdr->cap_cells = cap_cells;
}

__global__ void __launch_bounds__(256) grid_count_kernel(const float* __restrict__ verts, const int* __restrict__ tris,
                                                         int nt, GridHdr* hdr, int* __restrict__ counts,
                                                         int* __restrict__ over) {
  const GridHdr h = *hdr;
  float tau = 0.f;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    double g[3];
    const double rho = tri_centroid(verts, tris, t, g);
    if (!(rho <= h.c)) {  // big (or non-finite) triangles: scanned by every query
      over[atomicAdd(&hdr->n_over, 1)] = t;
    } else {
      atomicAdd(counts + cell_of(h, g), 1);
      tau = fmaxf(tau, __double2float_ru(rho));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) tau = fmaxf(tau, __shfl_xor_sync(0xffffffffu, tau, o));
  if ((threadIdx.x & 31) == 0 && tau > 0.f) atomicMax(&hdr->tau_key, float_key(tau));
}

__global__ void __launch_bounds__(256) grid_fill_kernel(const float* __restrict__ verts, const int* __restrict__ tris,
                                                        int nt, const GridHdr* __restrict__ hdr, int* __restrict__ counts,
                                                        const int* __restrict__ cell_start, int* __restrict__ sorted) {
  const GridHdr h = *hdr;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < nt; t += gridDim.x * blockDim.x) {
    double g[3];
    const double rho = tri_centroid(verts, tris, t, g);
    if (!(rho <= h.c)) continue;
    const int cell = cell_of(h, g);
    sorted[cell_start[cell] + atomicSub(counts + cell, 1) - 1] = t;  // any order inside a cell: the query ranks (d2, id)
  }
}

constexpr int kQueryThreads = 128;
constexpr int kQueryList = 4096;  // triangle ids gathered per shell before they are tested (balances the lanes)

// One block per landmark.  Per shell: the threads walk the shell's cells and copy the triangle ids of the non-empty ones
// into one shared list (cells hold very different numbers of triangles, and only ~10 % of a shell's cells touch the
// surface); then the list is tested with an even split over the threads.
__global__ void __launch_bounds__(kQueryThreads) grid_query_kernel(
    const float* __restrict__ verts, const int* __restrict__ tris, const GridHdr* __restrict__ hdr,
    const int* __restrict__ cell_start, const int* __restrict__ sorted, const int* __restrict__ over,
    const double* __restrict__ lm, double* __restrict__ out, int* __restrict__ out_tri, int* __restrict__ out_stats,
    int* __restrict__ handed_back) {
  __shared__ int s_list[kQueryList];
  __shared__ int s_total;
  __shared__ double s_best[kQueryThreads / 32];
  __shared__ int s_bt[kQueryThreads / 32], s_tests[kQueryThreads / 32];
  const int l = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const GridHdr h = *hdr;
  const double p[3] = {lm[3 * l], lm[3 * l + 1], lm[3 * l + 2]};
  double best = INFINITY;
  int bt = 0x7fffffff, n_tests = 0;
  auto test = [&](int t) {
    const double d = tri_dist2(verts, tris, t, p);
    if (d < best || (d == best && t < bt && d < INFINITY)) { best = d; bt = t; }  // like the scan: inf never wins
    ++n_tests;
  };
  for (int i = tid; i < h.n_over; i += kQueryThreads) test(over[i]);

  int ci[3], r_min = 0, r_max = 0;
  double margin = 0.5;
  bool finite = true;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double u = (p[i] - h.mn[i]) * h.inv_c;
    finite = finite && (u == u);
    u = fmin(fmax(u, -1.0e8), 1.0e8);  // clamping only shortens the lower bound below
    const double f = floor(u);
    ci[i] = static_cast<int>(f);
    margin = fmin(margin, fmin(u - f, f + 1.0 - u));
    r_min = max(r_min, ci[i] < 0 ? -ci[i] : (ci[i] > h.dim[i] - 1 ? ci[i] - (h.dim[i] - 1) : 0));
    r_max = max(r_max, max(ci[i], h.dim[i] - 1 - ci[i]));
  }
  const double tau = h.tau_key ? static_cast<double>(key_float(h.tau_key)) * (1.0 + 1e-6) : 0.0;
  int shells = 0;
  bool exhaustive = !finite;  // every decision below is uniform over the block
  for (int r = r_min; r <= r_max && !exhaustive; ++r, ++shells) {
    if (shells >= kMaxShells) { exhaustive = true; break; }
    // the shell = surface of the (2r+1)^3 box of cells: two full z faces, then the square's perimeter on the levels between
    const int side = 2 * r + 1, face = side * side, ring = 8 * r;
    const long long total_ll = r == 0 ? 1 : 2ll * face + static_cast<long long>(side - 2) * ring;
    if (total_ll > 8192) { exhaustive = true; break; }  // landmark cell > 18 cells outside the grid: far from any triangle
    const int total = static_cast<int>(total_ll);
    if (tid == 0) s_total = 0;
    __syncthreads();
    for (int j = tid; j < total; j += kQueryThreads) {
      int dx, dy, dz;
      if (j < 2 * face) {
        const int jj = j < face ? j : j - face;
        dz = j < face ? -r : r;
        dx = jj % side - r;
        dy = jj / side - r;
      } else {
        const int k = j - 2 * face, m = k % ring;
        dz = k / ring - r + 1;
        if (m < 2 * side) {
          dx = (m < side ? m : m - side) - r;
          dy = m < side ? -r : r;
        } else {
          const int mm = m - 2 * side;
          dx = mm / (side - 2) ? r : -r;
          dy = mm % (side - 2) - r + 1;
        }
      }
      const int x = ci[0] + dx, y = ci[1] + dy, z = ci[2] + dz;
      if (x < 0 || y < 0 || z < 0 || x >= h.dim[0] || y >= h.dim[1] || z >= h.dim[2]) continue;
      const int cell = (z * h.dim[1] + y) * h.dim[0] + x;
      const int b = cell_start[cell], cnt = cell_start[cell + 1] - b;
      if (cnt <= 0) continue;
      const int pos = atomicAdd(&s_total, cnt);
      if (pos + cnt <= kQueryList) {
        for (int k = 0; k < cnt; ++k) s_list[pos + k] = sorted[b + k];
      } else {  // list full: mark the part of the reservation that is inside the list and test this cell directly
        for (int k = pos; k < kQueryList; ++k) s_list[k] = -1;
        for (int k = 0; k < cnt; ++k) test(sorted[b + k]);
      }
    }
    __syncthreads();
    const int n_list = min(s_total, kQueryList);
    for (int i = tid; i < n_list; i += kQueryThreads) {
      const int t = s_list[i];
      if (t >= 0) test(t);
    }
    double wbest = best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wbest = fmin(wbest, __shfl_xor_sync(0xffffffffu, wbest, o));
    if (lane == 0) s_best[warp] = wbest;
    __syncthreads();
    wbest = fmin(fmin(s_best[0], s_best[1]), fmin(s_best[2], s_best[3]));
    __syncthreads();
    // every unvisited binned triangle has its centroid >= c (r + margin) away along some axis
    const double lb = h.c * (r + margin) * (1.0 - 1e-9) - 1e-9 * h.c - tau;
    if (lb > 0.0 && wbest < lb * lb) break;
  }
  if (exhaustive) {  // far from the surface (in cells) or non-finite: the (L, splits) scan kernels that follow do this one
    if (tid == 0) {
      handed_back[l] = 1;
      if (out_stats) { out_stats[2 * l] = h.nt; out_stats[2 * l + 1] = -1; }
    }
    return;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double od = __shfl_xor_sync(0xffffffffu, best, o);
    const int ot = __shfl_xor_sync(0xffffffffu, bt, o);
    if (od < best || (od == best && ot < bt)) { best = od; bt = ot; }
    n_tests += __shfl_xor_sync(0xffffffffu, n_tests, o);
  }
  if (lane == 0) { s_best[warp] = best; s_bt[warp] = bt; s_tests[warp] = n_tests; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < kQueryThreads / 32; ++w) {
      if (s_best[w] < best || (s_best[w] == best && s_bt[w] < bt)) { best = s_best[w]; bt = s_bt[w]; }
      n_tests += s_tests[w];
    }
    double q[3] = {p[0], p[1], p[2]};
    if (bt != 0x7fffffff) tri_closest(verts, tris, bt, p, q);
    out[3 * l] = q[0]; out[3 * l + 1] = q[1]; out[3 * l + 2] = q[2];
    if (out_tri) out_tri[l] = bt;
    if (out_stats) { out_stats[2 * l] = n_tests; out_stats[2 * l + 1] = shells; }
    handed_back[l] = 0;
  }
}

}  // namespace

size_t snap_grid_bytes(int nt) { return nt > 0 ? grid_layout(nt).total : 0; }

int snap_grid_build(const float* verts, const int* tris, int nt, void* grid, size_t grid_bytes, cudaStream_t s) {
  MVLM_REQUIRE(verts && tris && grid, "snap grid: null pointer");
  MVLM_REQUIRE(nt > 0, "snap grid: bad sizes");
  const GridLayout g = grid_layout(nt);
  MVLM_REQUIRE(grid_bytes >= g.total, "snap grid: buffer too small");
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(grid) & 15) == 0, "snap grid: buffer must be 16-byte aligned");
  uint8_t* base = static_cast<uint8_t*>(grid);
  GridHdr* hdr = reinterpret_cast<GridHdr*>(base);
  int* counts = reinterpret_cast<int*>(base + g.counts);
  int* cell_start = reinterpret_cast<int*>(base + g.cell_start);
  int* block_sums = reinterpret_cast<int*>(base + g.block_sums);
  int* sorted = reinterpret_cast<int*>(base + g.sorted);
  int* over = reinterpret_cast<int*>(base + g.over);
  MVLM_CHECK_CUDA(cudaMemsetAsync(base, 0, g.cell_start, s));  // header + counts
  const int blocks = min(ceil_div(nt, 256), 4 * sm_count());
  grid_bounds_kernel<<<blocks, 256, 0, s>>>(verts, tris, nt, hdr);
  grid_setup_kernel<<<1, 1, 0, s>>>(hdr, nt, g.cap_cells);
  grid_count_kernel<<<blocks, 256, 0, s>>>(verts, tris, nt, hdr, counts, over);
  exclusive_scan(counts, g.cap_cells, block_sums, cell_start, cell_start + g.cap_cells, s);
  grid_fill_kernel<<<blocks, 256, 0, s>>>(verts, tris, nt, hdr, counts, cell_start, sorted);
  count_launch(7);
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

size_t snap_grid_query_workspace_bytes(int l, int nt) {
  return snap_workspace_bytes(l, nt) + (static_cast<size_t>(l) * sizeof(int) + 63) / 64 * 64;
}

int snap_grid_query(const float* verts, const int* tris, int nt, const void* grid, size_t grid_bytes, const double* lm,
                    int l, void* workspace, size_t workspace_bytes, double* out, int* out_tri, int* out_stats,
                    cudaStream_t s) {
  MVLM_REQUIRE(verts && tris && grid && lm && out && workspace, "snap grid: null pointer");
  MVLM_REQUIRE(nt > 0 && l > 0, "snap grid: bad sizes");
  const GridLayout g = grid_layout(nt);
  MVLM_REQUIRE(grid_bytes >= g.total, "snap grid: buffer too small");
  MVLM_REQUIRE(workspace_bytes >= snap_grid_query_workspace_bytes(l, nt), "snap grid: workspace too small");
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, "snap grid: workspace must be 8-byte aligned");
  const uint8_t* base = static_cast<const uint8_t*>(grid);
  int* handed_back = reinterpret_cast<int*>(static_cast<uint8_t*>(workspace) + snap_workspace_bytes(l, nt));
  double* part = static_cast<double*>(workspace);
  grid_query_kernel<<<l, kQueryThreads, 0, s>>>(verts, tris, reinterpret_cast<const GridHdr*>(base),
                                      reinterpret_cast<const int*>(base + g.cell_start),
                                      reinterpret_cast<const int*>(base + g.sorted),
                                      reinterpret_cast<const int*>(base + g.over), lm, out, out_tri, out_stats,
                                      handed_back);
  count_launch(1);
  MVLM_CHECK_CUDA(cudaGetLastError());
  // landmarks the walk gave up on (more than kMaxShells cells from the surface, non-finite): the full scan, spread over
  // (L, splits) blocks; blocks of the other landmarks return at once
  const SnapMesh mesh = {verts, tris, nt};
  return snap_scan_launch(&mesh, 1, lm, l, part, out, out_tri, handed_back, s);
}

int snap_meshes_launch(const SnapMesh* meshes, const void* const* grids, int n_scans, const double* lm, int l,
                       void* workspace, size_t workspace_bytes, double* out, int* out_tri, cudaStream_t s) {
  const int rc = check_meshes(meshes, n_scans);
  if (rc != MVLM_OK) return rc;
  MVLM_REQUIRE(lm && out && workspace && l > 0, "snap: null pointer");
  MVLM_REQUIRE(workspace_bytes >= snap_meshes_workspace_bytes(meshes, n_scans, l), "snap: workspace too small");
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, "snap: workspace must be 8-byte aligned");
  int max_nt = 0, n_grids = 0;
  for (int i = 0; i < n_scans; ++i) {
    max_nt = max(max_nt, meshes[i].nt);
    n_grids += grids && grids[i] ? 1 : 0;
  }
  double* part = static_cast<double*>(workspace);
  int* only = nullptr;
  if (n_grids > 0) {
    // scans without a grid: every landmark goes to the scan kernel (any non-zero int); scans with one: the landmarks
    // their query hands back
    only = reinterpret_cast<int*>(static_cast<uint8_t*>(workspace) + snap_workspace_bytes(l * n_scans, max_nt));
    MVLM_CHECK_CUDA(cudaMemsetAsync(only, 0x01, static_cast<size_t>(l) * n_scans * sizeof(int), s));
    for (int i = 0; i < n_scans; ++i) {
      if (!grids || !grids[i]) continue;
      const uint8_t* base = static_cast<const uint8_t*>(grids[i]);
      const GridLayout g = grid_layout(meshes[i].nt);
      const size_t o = static_cast<size_t>(i) * l;
      grid_query_kernel<<<l, kQueryThreads, 0, s>>>(meshes[i].verts, meshes[i].tris, reinterpret_cast<const GridHdr*>(base),
                                                    reinterpret_cast<const int*>(base + g.cell_start),
                                                    reinterpret_cast<const int*>(base + g.sorted),
                                                    reinterpret_cast<const int*>(base + g.over), lm + 3 * o, out + 3 * o,
                                                    out_tri ? out_tri + o : nullptr, nullptr, only + o);
      count_launch(1);
    }
    MVLM_CHECK_CUDA(cudaGetLastError());
  }
  return snap_scan_launch(meshes, n_scans, lm, l, part, out, out_tri, only, s);
}

// debug: dims[3], n_over, cell edge, largest binned radius (synchronises the stream)
int snap_grid_describe(const void* grid, int* dims_nover, double* edge_tau, cudaStream_t s) {
  MVLM_REQUIRE(grid && dims_nover && edge_tau, "snap grid: null pointer");
  GridHdr h;
  MVLM_CHECK_CUDA(cudaMemcpyAsync(&h, grid, sizeof(h), cudaMemcpyDeviceToHost, s));
  MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
  for (int i = 0; i < 3; ++i) dims_nover[i] = h.dim[i];
  dims_nover[3] = h.n_over;
  edge_tau[0] = h.c;
  unsigned int k = h.tau_key;
  float tau = 0.f;
  if (k) {
    k ^= (k >> 31) ? 0x80000000u : 0xffffffffu;
    memcpy(&tau, &k, 4);
  }
  edge_tau[1] = tau;
  return MVLM_OK;
}

}  // namespace mvlm
