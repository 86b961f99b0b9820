// Per-landmark robust consensus: heat-value line filter, seeded multi-hypothesis RANSAC over
// view rays, least-squares closest point to the inlier lines.
//
// Replaces (reference src/mvlm/utils/estimator3d.py and utils3d.py):
//   filter_lines_based_on_heatmap_value_using_quantiles / _absolute_value  estimator3d.py:140-155
//   compute_intersection_between_lines (normal equations + pinv)            utils3d.py:99-124
//   compute_intersection_between_lines_ransac                               estimator3d.py:92-137
//   estimate_landmarks_from_lines                                           estimator3d.py:158-183
// The reference evaluates ONE hypothesis of 8 lines drawn with replacement from the unseeded
// global np.random (:105; the iteration loop is commented out, :103).  Here the hypothesis list is
// an explicit (L,H,8) uint32 table shared with the oracle (line index = draw mod n_lines); H=1 with
// the reference's own draw reproduces the reference.  Selection rule over hypotheses = the
// commented-out loop's: first strict minimum of the mean squared inlier distance.
//
// Kernels (all fp64; compiled with --fmad=false to round like numpy):
// Several scans of one pass run in the same three launches: grid axis z (prepare: y) is the scan, peaks / rays are
// read with the pass's view stride ((L, S*V, 3), scan s at views [s*V, (s+1)*V)), every per-landmark slot of the
// workspace and the outputs is (S, L, ...).  A scan's result does not depend on the other scans nor on `splits`.
//
//   consensus_prepare     one block per (landmark, scan): np.quantile('linear', float32) threshold, strict
//                         `>` mask, order-preserving compaction, per-line normal-equation terms
//                         M_i = n n^T - I and M_i a_i, LSQ over all kept lines (the fallback).
//   consensus_hypotheses  grid (L, splits): lines of the landmark staged in shared memory, one THREAD
//                         per hypothesis (8-line LSQ -> one pass over all lines: inlier test + count +
//                         normal-equation sums -> inlier refit -> score pass), warp-shuffle + shared
//                         memory reduction of the lexicographic (error, hypothesis) minimum.
//   consensus_finalize    lexicographic (error, hypothesis) minimum over splits, fallbacks.
//   consensus_report      (only when report outputs are given) one block per (landmark, scan): status, inlier mask
//                         in view order, counts, rms and covariance of the final fit (DESIGN.md 7h).
#include "common.cuh"
#include "stages.cuh"

namespace mvlm {

namespace {

constexpr int kLineDoubles = 16;  // a[3] b[3] M[6]={xx,yy,zz,xy,xz,yz} Ma[3] |b-a|
constexpr int kMaxViews = 1024;
constexpr int kPartDoubles = 5;   // err, hyp, p[3]
constexpr double kNoFit = 100000000.0;  // estimator3d.py:95

// Jacobi eigen-decomposition of the symmetric 3x3 matrix S6 = {xx,yy,zz,xy,xz,yz}: eigenvalues lam[k], eigenvector k
// in column k of v.
__device__ __forceinline__ void sym3_jacobi(const double* S6, double lam[3], double v[3][3]) {
  double a[3][3] = {{S6[0], S6[3], S6[4]}, {S6[3], S6[1], S6[5]}, {S6[4], S6[5], S6[2]}};
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int k = 0; k < 3; ++k) v[r][k] = r == k ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 12; ++sweep) {
    const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
    const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
    if (off <= 1e-34 * diag) break;  // eigenvalues converged far below double rounding
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int pi = k == 2 ? 1 : 0;
      const int qi = k == 0 ? 1 : 2;
      const double apq = a[pi][qi];
      if (apq == 0.0) continue;
      const double theta = (a[qi][qi] - a[pi][pi]) / (2.0 * apq);
      const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      const double cs = 1.0 / sqrt(t * t + 1.0);
      const double sn = t * cs;
      for (int r = 0; r < 3; ++r) {  // A <- A J
        const double arp = a[r][pi], arq = a[r][qi];
        a[r][pi] = cs * arp - sn * arq;
        a[r][qi] = sn * arp + cs * arq;
      }
      for (int r = 0; r < 3; ++r) {  // A <- J^T A
        const double apr = a[pi][r], aqr = a[qi][r];
        a[pi][r] = cs * apr - sn * aqr;
        a[qi][r] = sn * apr + cs * aqr;
      }
      for (int r = 0; r < 3; ++r) {
        const double vrp = v[r][pi], vrq = v[r][qi];
        v[r][pi] = cs * vrp - sn * vrq;
        v[r][qi] = sn * vrp + cs * vrq;
      }
    }
  }
  lam[0] = a[0][0]; lam[1] = a[1][1]; lam[2] = a[2][2];
}

// Eigenvalues at or below this are dropped as singular (np.linalg.pinv default rcond, utils3d.py:123).
__device__ __forceinline__ double sym3_cut(const double lam[3]) {
  return 1e-15 * fmax(fabs(lam[0]), fmax(fabs(lam[1]), fabs(lam[2])));
}

// Minimum-norm solve of the symmetric 3x3 system S p = c via the Jacobi eigen-decomposition, singular values at or
// below sym3_cut dropped.
__device__ void sym3_pinv_solve(const double* S6, const double* c, double* p) {
  double lam[3], v[3][3];
  sym3_jacobi(S6, lam, v);
  const double cut = sym3_cut(lam);
  p[0] = p[1] = p[2] = 0.0;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if (fabs(lam[k]) > cut) {
      const double proj = (v[0][k] * c[0] + v[1][k] * c[1] + v[2][k] * c[2]) / lam[k];
      p[0] += proj * v[0][k];
      p[1] += proj * v[1][k];
      p[2] += proj * v[2][k];
    }
  }
}

// (|(p-a) x (p-b)| / |b-a|)^2   estimator3d.py:109-111
__device__ __forceinline__ double line_sqdist(const double* p, const double* ln) {
  const double ax = p[0] - ln[0], ay = p[1] - ln[1], az = p[2] - ln[2];
  const double bx = p[0] - ln[3], by = p[1] - ln[4], bz = p[2] - ln[5];
  const double cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
  const double top = sqrt((cx * cx + cy * cy) + cz * cz);
  const double d = top / ln[15];  // |b-a| = np.linalg.norm(bottom), precomputed per line
  return d * d;
}

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

struct Layout {
  double* lines;  // S * L * V * 16
  double* p_all;  // S * L * 3
  double* part;   // S * L * splits * 5
  int* nl;        // S * L
};

// L: landmarks x scans of the pass
__host__ __device__ inline Layout carve(void* ws, int L, int V, int splits) {
  Layout o;
  double* d = static_cast<double*>(ws);
  o.lines = d;
  d += static_cast<size_t>(L) * V * kLineDoubles;
  o.p_all = d;
  d += static_cast<size_t>(L) * 3;
  o.part = d;
  d += static_cast<size_t>(L) * splits * kPartDoubles;
  o.nl = reinterpret_cast<int*>(d);
  return o;
}

// Row of landmark l's views of scan s in the (L, S*V, 3) peaks / rays.
__device__ __forceinline__ size_t view_row(const ConsensusArgs& g, int l, int s) {
  return static_cast<size_t>(l) * g.n_scans * g.v + static_cast<size_t>(s) * g.v;
}

// Heat-value line filter of one (landmark, scan) slot, called by the whole block: keep[i] = 1 for the views i whose
// value is strictly above the quantile / absolute threshold.  vals (V floats), keep (V bytes), sel (2 floats) and
// any_nan are the caller's shared memory; returns after a barrier, with keep complete.
__device__ void filter_keep_mask(const ConsensusArgs& g, size_t row, float* vals, unsigned char* keep, float* sel,
                                 int* any_nan) {
  const int V = g.v, tid = threadIdx.x;
  if (tid == 0) { *any_nan = 0; sel[0] = sel[1] = 0.f; }
  __syncthreads();
  for (int i = tid; i < V; i += blockDim.x) {
    const float x = g.peaks[(row + i) * 3 + 2];
    vals[i] = x;
    if (x != x) *any_nan = 1;
  }
  __syncthreads();
  float thr;
  if (g.mode == 1) {
    thr = g.threshold_absolute;
  } else {
    // np.quantile(values float32, q python float, method='linear'): q and the virtual index are
    // float32 (numpy >= 2.0 matches q to the array dtype), _lerp in float32.
    const float q32 = static_cast<float>(g.threshold_quantile);
    const float virt = static_cast<float>(V - 1) * q32;
    int lo = static_cast<int>(floorf(virt));
    int hi = lo + 1;
    const float t = virt - static_cast<float>(lo);
    if (virt >= static_cast<float>(V - 1)) { lo = V - 1; hi = V - 1; }
    if (virt < 0.f) { lo = 0; hi = 0; }
    for (int i = tid; i < V; i += blockDim.x) {
      const float x = vals[i];
      int rank = 0;
      for (int j = 0; j < V; ++j) {
        const float y = vals[j];
        rank += (y < x || (y == x && j < i)) ? 1 : 0;
      }
      if (rank == lo) sel[0] = x;
      if (rank == hi) sel[1] = x;
    }
    __syncthreads();
    const float a = sel[0], b = sel[1];
    const float diff = b - a;
    thr = a + diff * t;
    if (t >= 0.5f) thr = b - diff * (1.0f - t);
    if (*any_nan) thr = NAN;  // np.quantile -> nan -> every comparison False
  }
  for (int i = tid; i < V; i += blockDim.x) keep[i] = vals[i] > thr ? 1 : 0;
  __syncthreads();
}

__global__ void __launch_bounds__(256) consensus_prepare_kernel(ConsensusArgs g, Layout ws) {
  __shared__ float vals[kMaxViews];
  __shared__ unsigned char keep[kMaxViews];
  __shared__ float sel[2];
  __shared__ int any_nan;
  __shared__ double red[9][8];
  const int V = g.v, tid = threadIdx.x;
  const int sl = blockIdx.y * g.l + blockIdx.x;  // (scan, landmark) slot
  const size_t row = view_row(g, blockIdx.x, blockIdx.y);
  filter_keep_mask(g, row, vals, keep, sel, &any_nan);
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  int n_kept = 0;
  for (int i = 0; i < V; ++i) n_kept += keep[i];  // every thread: tiny V
  for (int i = tid; i < V; i += blockDim.x) {
    if (!keep[i]) continue;
    int pos = 0;
    for (int j = 0; j < i; ++j) pos += keep[j];
    const double* a = g.starts + (row + i) * 3;
    const double* b = g.ends + (row + i) * 3;
    const double sx = b[0] - a[0], sy = b[1] - a[1], sz = b[2] - a[2];
    const double nrm = sqrt((sx * sx + sy * sy) + sz * sz);
    const double nx = sx / nrm, ny = sy / nrm, nz = sz / nrm;
    double* ln = ws.lines + (static_cast<size_t>(sl) * V + pos) * kLineDoubles;
    ln[0] = a[0]; ln[1] = a[1]; ln[2] = a[2];
    ln[3] = b[0]; ln[4] = b[1]; ln[5] = b[2];
    const double mxx = nx * nx - 1.0, myy = ny * ny - 1.0, mzz = nz * nz - 1.0;
    const double mxy = nx * ny, mxz = nx * nz, myz = ny * nz;
    ln[6] = mxx; ln[7] = myy; ln[8] = mzz; ln[9] = mxy; ln[10] = mxz; ln[11] = myz;
    ln[12] = (a[0] * mxx + a[1] * mxy) + a[2] * mxz;
    ln[13] = (a[0] * mxy + a[1] * myy) + a[2] * myz;
    ln[14] = (a[0] * mxz + a[1] * myz) + a[2] * mzz;
    ln[15] = nrm;
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] += ln[6 + k];
  }
  const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const double s = warp_sum(acc[k]);
    if (lane == 0) red[k][warp] = s;
  }
  __syncthreads();
  if (tid == 0) {
    double S[9];
    for (int k = 0; k < 9; ++k) {
      double s = 0.0;
      for (int w = 0; w < 8; ++w) s += red[k][w];
      S[k] = s;
    }
    double p[3];
    sym3_pinv_solve(S, S + 6, p);
    ws.p_all[3 * sl] = p[0]; ws.p_all[3 * sl + 1] = p[1]; ws.p_all[3 * sl + 2] = p[2];
    ws.nl[sl] = n_kept;
    if (g.out_nlines) g.out_nlines[sl] = n_kept;
  }
}

// One THREAD per hypothesis (the lines of the landmark are broadcast reads from shared memory):
//   8-line LSQ -> one pass over all lines (inlier test, count, normal-equation sums of the inliers)
//   -> if count > n/3: refit, second pass (mean squared distance of the inliers to the refit point).
__global__ void __launch_bounds__(256) consensus_hyp_kernel(ConsensusArgs g, Layout ws, int splits, int chunk) {
  extern __shared__ double sl[];  // n * 16
  __shared__ double wbest[8][kPartDoubles];
  const int l = blockIdx.x, split = blockIdx.y;
  const int slot = blockIdx.z * g.l + l;  // (scan, landmark) slot
  const int n = ws.nl[slot];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  double* part = ws.part + (static_cast<size_t>(slot) * splits + split) * kPartDoubles;
  if (n < 3) {  // plain LSQ, handled by finalize
    if (tid == 0) { part[0] = kNoFit; part[1] = -1.0; part[2] = part[3] = part[4] = 0.0; }
    return;
  }
  const double* gl = ws.lines + static_cast<size_t>(slot) * g.v * kLineDoubles;
  const unsigned int* draws_l = g.draws + static_cast<size_t>(blockIdx.z) * g.draws_scan_stride +
                                static_cast<size_t>(l) * g.n_hyp * 8;
  for (int i = tid; i < n * kLineDoubles; i += blockDim.x) sl[i] = gl[i];
  __syncthreads();
  const int h_begin = split * chunk;
  const int h_end = min(g.n_hyp, h_begin + chunk);
  const double need = static_cast<double>(n) / 3.0;  // d = n_lines / 3, :100
  const double thres = g.dist_thres;
  double best_err = kNoFit, best_h = -1.0, bp0 = 0.0, bp1 = 0.0, bp2 = 0.0;
  for (int h = h_begin + tid; h < h_end; h += blockDim.x) {
    // --- 8-line LSQ (:105-107)
    double s9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    const uint4* dr = reinterpret_cast<const uint4*>(draws_l + static_cast<size_t>(h) * 8);
    const uint4 d0 = __ldg(dr), d1 = __ldg(dr + 1);
    const unsigned int draws[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const double* ln = sl + static_cast<size_t>(draws[q] % static_cast<unsigned int>(n)) * kLineDoubles;
#pragma unroll
      for (int k = 0; k < 9; ++k) s9[k] += ln[6 + k];
    }
    double p[3];
    sym3_pinv_solve(s9, s9 + 6, p);
    // --- inliers (:109-114) and their normal-equation sums in one pass
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int cnt = 0;
    for (int i = 0; i < n; ++i) {
      const double* ln = sl + static_cast<size_t>(i) * kLineDoubles;
      if (line_sqdist(p, ln) < thres) {
        ++cnt;
#pragma unroll
        for (int k = 0; k < 9; ++k) acc[k] += ln[6 + k];
      }
    }
    if (static_cast<double>(cnt) > need) {
      // --- refit on the inliers and score (:116-125)
      double p2[3];
      sym3_pinv_solve(acc, acc + 6, p2);
      double ds = 0.0;
      for (int i = 0; i < n; ++i) {
        const double* ln = sl + static_cast<size_t>(i) * kLineDoubles;
        if (line_sqdist(p, ln) < thres) ds += line_sqdist(p2, ln);
      }
      const double err = ds / static_cast<double>(cnt);
      if (err < best_err) {  // strict <, hypotheses visited in increasing order
        best_err = err; best_h = h; bp0 = p2[0]; bp1 = p2[1]; bp2 = p2[2];
      }
    }
  }
  // block reduction: lexicographic (error, hypothesis) minimum -> first strict minimum over the whole range
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double oe = __shfl_xor_sync(0xffffffffu, best_err, o), oh = __shfl_xor_sync(0xffffffffu, best_h, o);
    const double o0 = __shfl_xor_sync(0xffffffffu, bp0, o), o1 = __shfl_xor_sync(0xffffffffu, bp1, o);
    const double o2 = __shfl_xor_sync(0xffffffffu, bp2, o);
    const bool take = oh >= 0.0 && (best_h < 0.0 || oe < best_err || (oe == best_err && oh < best_h));
    if (take) { best_err = oe; best_h = oh; bp0 = o0; bp1 = o1; bp2 = o2; }
  }
  if (lane == 0) {
    wbest[warp][0] = best_err; wbest[warp][1] = best_h; wbest[warp][2] = bp0; wbest[warp][3] = bp1; wbest[warp][4] = bp2;
  }
  __syncthreads();
  if (tid == 0) {
    int bw = -1;
    for (int w = 0; w < 8; ++w) {
      if (wbest[w][1] < 0.0) continue;
      if (bw < 0 || wbest[w][0] < wbest[bw][0] || (wbest[w][0] == wbest[bw][0] && wbest[w][1] < wbest[bw][1])) bw = w;
    }
    if (bw < 0) { part[0] = kNoFit; part[1] = -1.0; part[2] = part[3] = part[4] = 0.0; }
    else for (int k = 0; k < kPartDoubles; ++k) part[k] = wbest[bw][k];
  }
}

// Split holding a slot's winning hypothesis: the lexicographic (error, hypothesis) minimum over the splits' partial
// results; -1 when no split accepted one.  part = the slot's `splits` records of kPartDoubles.
__device__ __forceinline__ int winning_split(const double* part, int splits) {
  int bs = -1;
  for (int s = 0; s < splits; ++s) {
    const double* q = part + s * kPartDoubles;
    if (q[1] < 0.0) continue;
    if (bs < 0 || q[0] < part[bs * kPartDoubles] ||
        (q[0] == part[bs * kPartDoubles] && q[1] < part[bs * kPartDoubles + 1]))
      bs = s;
  }
  return bs;
}

__global__ void consensus_finalize_kernel(ConsensusArgs g, Layout ws, int splits) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;  // (scan, landmark) slot
  if (l >= g.l * g.n_scans) return;
  const int n = ws.nl[l];
  const double* part = ws.part + static_cast<size_t>(l) * splits * kPartDoubles;
  const int bs = n >= 3 ? winning_split(part, splits) : -1;
  double* o = g.out_landmarks + 3 * l;
  if (bs >= 0) {
    const double* q = part + bs * kPartDoubles;
    o[0] = q[2]; o[1] = q[3]; o[2] = q[4];
    g.out_errors[l] = q[0];
  } else {
    o[0] = ws.p_all[3 * l]; o[1] = ws.p_all[3 * l + 1]; o[2] = ws.p_all[3 * l + 2];
    // < 3 lines: plain LSQ, contributes 0 (:174-176); RANSAC without an accepted hypothesis: LSQ
    // over all lines, error stays 1e8 (:131-133)
    g.out_errors[l] = n < 3 ? 0.0 : kNoFit;
  }
}

// One block per (landmark, scan) slot, after finalize, on the same workspace: which lines the final fit used and how
// well they agree.  The filter and the winner are the ones prepare and finalize computed (same functions, same
// inputs); the winner's 8-line point, inlier test, refit and squared distances repeat consensus_hyp_kernel's
// arithmetic in its order, so the inlier set is the one the hypothesis kernel scored and the refit point is
// out_landmarks bit for bit (status 0: rms^2 sums exactly what out_errors sums).  The per-line sums run on one thread
// in line order; every other thread only rebuilds the filter and writes the mask.
__global__ void __launch_bounds__(256) consensus_report_kernel(ConsensusArgs g, Layout ws, int splits,
                                                               ConsensusReport r) {
  __shared__ float vals[kMaxViews];
  __shared__ unsigned char keep[kMaxViews];
  __shared__ unsigned char used[kMaxViews];  // by compacted line position
  __shared__ short pos_of[kMaxViews];        // compacted line position of each kept view
  __shared__ float sel[2];
  __shared__ int any_nan;
  const int V = g.v, tid = threadIdx.x;
  const int slot = blockIdx.y * g.l + blockIdx.x;  // (scan, landmark) slot
  filter_keep_mask(g, view_row(g, blockIdx.x, blockIdx.y), vals, keep, sel, &any_nan);
  for (int i = tid; i < V; i += blockDim.x) {
    if (!keep[i]) continue;
    int pos = 0;
    for (int j = 0; j < i; ++j) pos += keep[j];
    pos_of[i] = static_cast<short>(pos);
  }
  const int n = ws.nl[slot];
  if (tid == 0) {
    const double* lines = ws.lines + static_cast<size_t>(slot) * V * kLineDoubles;
    const double* part = ws.part + static_cast<size_t>(slot) * splits * kPartDoubles;
    const int bs = n >= 3 ? winning_split(part, splits) : -1;
    double c[3];  // the consensus point
    int k;        // lines of the final fit
    signed char status;
    if (bs >= 0) {
      // --- the winner's 8-line LSQ, inliers and refit, as in consensus_hyp_kernel
      const int h = static_cast<int>(part[bs * kPartDoubles + 1]);
      const unsigned int* dr = g.draws + static_cast<size_t>(blockIdx.y) * g.draws_scan_stride +
                               (static_cast<size_t>(blockIdx.x) * g.n_hyp + h) * 8;
      double s9[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      for (int q = 0; q < 8; ++q) {
        const double* ln = lines + static_cast<size_t>(dr[q] % static_cast<unsigned int>(n)) * kLineDoubles;
#pragma unroll
        for (int j = 0; j < 9; ++j) s9[j] += ln[6 + j];
      }
      double p[3];
      sym3_pinv_solve(s9, s9 + 6, p);
      double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      k = 0;
      for (int i = 0; i < n; ++i) {
        const double* ln = lines + static_cast<size_t>(i) * kLineDoubles;
        used[i] = line_sqdist(p, ln) < g.dist_thres ? 1 : 0;
        if (used[i]) {
          ++k;
#pragma unroll
          for (int j = 0; j < 9; ++j) acc[j] += ln[6 + j];
        }
      }
      sym3_pinv_solve(acc, acc + 6, c);
      status = 0;
    } else {
      // --- no accepted hypothesis (status 1) or fewer than 3 lines (status 2): LSQ over every kept line
      for (int i = 0; i < n; ++i) used[i] = 1;
      k = n;
      c[0] = ws.p_all[3 * slot]; c[1] = ws.p_all[3 * slot + 1]; c[2] = ws.p_all[3 * slot + 2];
      status = n < 3 ? 2 : 1;
    }
    // --- squared distances of the used lines and J = sum (I - n n^T) = -sum M_i
    double ds = 0.0, J[6] = {0, 0, 0, 0, 0, 0};
    for (int i = 0; i < n; ++i) {
      if (!used[i]) continue;
      const double* ln = lines + static_cast<size_t>(i) * kLineDoubles;
      ds += line_sqdist(c, ln);
#pragma unroll
      for (int j = 0; j < 6; ++j) J[j] -= ln[6 + j];
    }
    r.status[slot] = status;
    r.n_inliers[slot] = k;
    r.rms[slot] = sqrt(ds / static_cast<double>(k));  // k = 0: NaN
    // covariance sigma^2 J^-1, sigma^2 = ds / (2k - 3): each line constrains the two directions across it
    double* cov = r.covariance + static_cast<size_t>(slot) * 9;
    double lam[3], v[3][3];
    sym3_jacobi(J, lam, v);
    const double cut = sym3_cut(lam);
    const bool full_rank = k >= 2 && fabs(lam[0]) > cut && fabs(lam[1]) > cut && fabs(lam[2]) > cut;
    const double s2 = ds / static_cast<double>(2 * k - 3);
    for (int a = 0; a < 3; ++a)
      for (int b = 0; b < 3; ++b)
        cov[3 * a + b] = full_rank ? s2 * (v[a][0] * v[b][0] / lam[0] + v[a][1] * v[b][1] / lam[1] +
                                           v[a][2] * v[b][2] / lam[2])
                                   : NAN;
  }
  __syncthreads();
  unsigned char* mask = r.inliers + static_cast<size_t>(slot) * V;
  for (int i = tid; i < V; i += blockDim.x) mask[i] = keep[i] ? used[pos_of[i]] : 0;
}

int pick_splits(int l, int n_hyp) {
  int splits = ceil_div(2 * sm_count(), l);
  const int max_splits = ceil_div(n_hyp, 256);  // at least one hypothesis per thread
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  return splits;
}

}  // namespace

size_t consensus_workspace_bytes(int l, int v, int n_hyp, int n_scans) {
  l *= n_scans;
  const int splits = pick_splits(l, n_hyp);
  size_t d = static_cast<size_t>(l) * v * kLineDoubles + static_cast<size_t>(l) * 3 +
             static_cast<size_t>(l) * splits * kPartDoubles;
  return d * sizeof(double) + static_cast<size_t>(l) * sizeof(int) + 64;
}

int consensus_launch(const ConsensusArgs& a, cudaStream_t s, const ConsensusReport* report) {
  MVLM_REQUIRE(a.peaks && a.starts && a.ends && a.draws && a.out_landmarks && a.out_errors && a.workspace,
               "consensus: null pointer");
  MVLM_REQUIRE(!report || (report->status && report->n_inliers && report->inliers && report->rms && report->covariance),
               "consensus: null report output");
  MVLM_REQUIRE(a.l > 0 && a.v > 0 && a.n_hyp > 0 && a.n_scans > 0 && a.n_scans <= 65535, "consensus: bad sizes");
  MVLM_REQUIRE(a.draws_scan_stride == 0 || a.draws_scan_stride == static_cast<size_t>(a.l) * a.n_hyp * 8,
               "consensus: draws are one shared (L,H,8) table or one (S,L,H,8) table");
  MVLM_REQUIRE(a.v <= kMaxViews, "consensus: at most %d views supported (got %d)", kMaxViews, a.v);
  MVLM_REQUIRE(a.mode == 0 || a.mode == 1, "consensus: Unknown mode for line matching in Estimator: %d", a.mode);
  MVLM_REQUIRE(a.workspace_bytes >= consensus_workspace_bytes(a.l, a.v, a.n_hyp, a.n_scans),
               "consensus: workspace too small");
  const int slots = a.l * a.n_scans;
  const int splits = pick_splits(slots, a.n_hyp);
  const int chunk = ceil_div(a.n_hyp, splits);
  Layout ws = carve(a.workspace, slots, a.v, splits);
  consensus_prepare_kernel<<<dim3(a.l, a.n_scans), 256, 0, s>>>(a, ws);
  const size_t smem = static_cast<size_t>(a.v) * kLineDoubles * sizeof(double);
  // more than 48 KB (over 384 views): the opt-in attribute is per device, so it is set on every such launch
  // (a host-side call of about a microsecond; the common cases stay below the limit)
  if (smem > 48 * 1024)
    MVLM_CHECK_CUDA(cudaFuncSetAttribute(consensus_hyp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         static_cast<int>(smem)));
  consensus_hyp_kernel<<<dim3(a.l, splits, a.n_scans), 256, smem, s>>>(a, ws, splits, chunk);
  consensus_finalize_kernel<<<ceil_div(slots, 128), 128, 0, s>>>(a, ws, splits);
  count_launch(3);
  if (report) {
    consensus_report_kernel<<<dim3(a.l, a.n_scans), 256, 0, s>>>(a, ws, splits, *report);
    count_launch(1);
  }
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

}  // namespace mvlm
