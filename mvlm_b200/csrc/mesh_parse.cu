// PLY / STL scan decoder on the GPU (opt-in alternative to the host loader mesh_loader.cu, which is the specification:
// the same arrays bit for bit).  The host parses only the PLY header, or checks the STL size rule, and the bytes of
// the file cross PCIe instead of the decoded arrays.
//
// Binary PLY (every element other than `face` of fixed size, `face` holding only its index list):
//   check   speculative fixed-stride layout: every face is assumed to be a triangle (record = count + 3 indices), which
//           the body length must match exactly.  One thread per face checks that its count is 3 and its indices are in
//           range; if every check passes the layout is proven by induction (record t starts where the thread looked
//           because records 0 .. t-1 are triangles).  Any failure sets the fallback flag: the file goes to the host
//           loader, which also reports its errors.
//   write   (phase 2) one thread per vertex record gathers x y z (and red green blue) with a byte swap for big-endian
//           files and the conversion to f32; one thread per face gathers its three indices.
// Binary STL, then the weld (exact-equality unique of the 96-bit corner keys, first-occurrence numbering):
//   decode  one thread per 50-byte facet record: its three corners
//   insert  one thread per corner: open-addressing hash table of corner indices (keys compared through the corners'
//           coordinates); an equal key already present takes atomicMin of the index, so every slot ends holding the
//           SMALLEST corner index of its key, whatever the order of the inserts.  NaN corners are not inserted.
//   leader  one thread per corner: its key's slot -> its leader (the first corner with that key; a NaN corner is its
//           own leader); first[i] = (leader == i)
//   scan    exclusive scan of first[] in corner order (scan.cuh): the vertex id of every leader = order of first
//           occurrence
//   facet   one thread per facet: the vertex ids of its corners, keep = three distinct ids; scan of keep[] (file order)
//   write   (phase 2) leaders scatter their coordinates to their vertex ids, kept facets to their triangle ids
// Capacity: the scans take 16.7M items, so 5.5M facets (16.7M corners); a larger STL is read on the host.
#include "../../include/mvlm_b200.h"
#include "common.cuh"
#include "mesh_format.cuh"
#include "scan.cuh"

namespace mvlm {
namespace {

using namespace mesh;

struct PlyLayout {
  long long v_off, f_off;  // byte offsets of the vertex / face element in the file
  int v_stride, f_stride;
  int nv, nf;
  int xo[3], xt[3];        // offsets within a vertex record and types of x y z
  int co[3];               // offsets of red green blue (uchar), -1: no colours
  int cnt_type, idx_type, cnt_size, idx_size;
  int big;
};

struct DevHdr {
  int fallback;
  int n_verts, n_tris;  // totals of the two weld scans
  PlyLayout ply;        // the layout of phase 1, read by phase 2's kernels
};

size_t round256(size_t b) { return (b + 255) / 256 * 256; }

struct StlLayout {
  bool fits;
  int nf, n, n_pad, f_pad;
  size_t slots;
  size_t bytes, hdr, pos, table, leader, first, vid, ids, keep, toff, block_sums, total;
};

StlLayout stl_layout(size_t n_bytes) {
  StlLayout L{};
  if (n_bytes < 84 || (n_bytes - 84) % 50 != 0) return L;
  const size_t nf = (n_bytes - 84) / 50;
  const size_t n = 3 * nf;
  const size_t n_pad = (n + kScanItems) / kScanItems * kScanItems;
  const size_t f_pad = (nf + kScanItems) / kScanItems * kScanItems;
  L.fits = nf > 0 && n_pad <= static_cast<size_t>(kScanItems) * kScanMaxBlocks;
  if (!L.fits) return L;
  L.nf = static_cast<int>(nf);
  L.n = static_cast<int>(n);
  L.n_pad = static_cast<int>(n_pad);
  L.f_pad = static_cast<int>(f_pad);
  L.slots = weld_table_slots(n);
  size_t o = 0;
  auto take = [&](size_t b) {
    const size_t at = o;
    o += round256(b);
    return at;
  };
  L.bytes = take(n_bytes);
  L.hdr = take(sizeof(DevHdr));
  L.pos = take(n * 12);
  L.table = take(L.slots * 4);
  L.leader = take(n * 4);
  L.first = take(n_pad * 4);
  L.vid = take(n_pad * 4);
  L.ids = take(n * 4);
  L.keep = take(f_pad * 4);
  L.toff = take(f_pad * 4);
  L.block_sums = take(kScanMaxBlocks * 4);
  L.total = o;
  return L;
}

size_t ply_workspace_bytes(size_t n_bytes) { return round256(n_bytes) + round256(sizeof(DevHdr)); }

// ---- PLY -------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) ply_check_kernel(const uint8_t* __restrict__ b, const PlyLayout L,
                                                        DevHdr* __restrict__ hdr) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t == 0) hdr->ply = L;
  if (t >= L.nf) return;
  const uint8_t* r = b + L.f_off + static_cast<long long>(t) * L.f_stride;
  bool ok = read_int(r, L.cnt_type, L.big) == 3;
  for (int j = 0; ok && j < 3; ++j) {
    const long long i = read_int(r + L.cnt_size + j * L.idx_size, L.idx_type, L.big);
    ok = i >= 0 && i < L.nv;
  }
  if (!ok) atomicOr(&hdr->fallback, 1);
}

__global__ void __launch_bounds__(256) ply_vertex_kernel(const uint8_t* __restrict__ b, const DevHdr* __restrict__ hdr,
                                                         float* __restrict__ verts, uint8_t* __restrict__ colors) {
  const PlyLayout& L = hdr->ply;
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= L.nv) return;
  const uint8_t* r = b + L.v_off + static_cast<long long>(v) * L.v_stride;
  for (int c = 0; c < 3; ++c) verts[3ll * v + c] = read_coord(r + L.xo[c], L.xt[c], L.big);
  if (colors)
    for (int c = 0; c < 3; ++c) colors[3ll * v + c] = r[L.co[c]];
}

__global__ void __launch_bounds__(256) ply_face_kernel(const uint8_t* __restrict__ b, const DevHdr* __restrict__ hdr,
                                                       int32_t* __restrict__ tris) {
  const PlyLayout& L = hdr->ply;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= L.nf) return;
  const uint8_t* r = b + L.f_off + static_cast<long long>(t) * L.f_stride + L.cnt_size;
  for (int j = 0; j < 3; ++j) tris[3ll * t + j] = static_cast<int32_t>(read_int(r + j * L.idx_size, L.idx_type, L.big));
}

// ---- STL + weld ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stl_decode_kernel(const uint8_t* __restrict__ b, int nf, float* __restrict__ pos) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nf) return;
  const uint8_t* r = b + 84 + 50ll * t + 12;  // skip the facet normal; records are only 2-byte aligned
  for (int j = 0; j < 9; ++j) pos[9ll * t + j] = read_coord(r + 4 * j, kFloat, false);
}

__device__ __forceinline__ bool same_key(const float* __restrict__ pos, int j, uint32_t kx, uint32_t ky, uint32_t kz) {
  return weld_bits(pos[3ll * j]) == kx && weld_bits(pos[3ll * j + 1]) == ky && weld_bits(pos[3ll * j + 2]) == kz;
}

__global__ void __launch_bounds__(256) weld_insert_kernel(const float* __restrict__ pos, int n, int* __restrict__ table,
                                                          unsigned int mask) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = pos[3ll * i], y = pos[3ll * i + 1], z = pos[3ll * i + 2];
  if (weld_is_nan(x, y, z)) return;
  const uint32_t kx = weld_bits(x), ky = weld_bits(y), kz = weld_bits(z);
  for (unsigned int s = weld_hash(kx, ky, kz) & mask;; s = (s + 1) & mask) {
    const int cur = atomicCAS(table + s, -1, i);
    if (cur == -1) return;
    if (same_key(pos, cur, kx, ky, kz)) {  // every index a slot ever holds has the same key
      atomicMin(table + s, i);
      return;
    }
  }
}

__global__ void __launch_bounds__(256) weld_leader_kernel(const float* __restrict__ pos, int n,
                                                          const int* __restrict__ table, unsigned int mask,
                                                          int* __restrict__ leader, int* __restrict__ first) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = pos[3ll * i], y = pos[3ll * i + 1], z = pos[3ll * i + 2];
  int l = i;
  if (!weld_is_nan(x, y, z)) {
    const uint32_t kx = weld_bits(x), ky = weld_bits(y), kz = weld_bits(z);
    for (unsigned int s = weld_hash(kx, ky, kz) & mask;; s = (s + 1) & mask) {
      const int cur = table[s];  // never empty before this key's slot: the key was inserted
      if (same_key(pos, cur, kx, ky, kz)) {
        l = cur;
        break;
      }
    }
  }
  leader[i] = l;
  first[i] = l == i ? 1 : 0;
}

__global__ void __launch_bounds__(256) weld_facet_kernel(const int* __restrict__ leader, const int* __restrict__ vid,
                                                         int nf, int* __restrict__ ids, int* __restrict__ keep) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nf) return;
  int v[3];
  for (int j = 0; j < 3; ++j) {
    v[j] = vid[leader[3ll * t + j]];
    ids[3ll * t + j] = v[j];
  }
  keep[t] = (v[0] != v[1] && v[1] != v[2] && v[0] != v[2]) ? 1 : 0;
}

__global__ void __launch_bounds__(256) weld_write_verts_kernel(const float* __restrict__ pos, const int* __restrict__ first,
                                                               const int* __restrict__ vid, int n, float* __restrict__ verts) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || !first[i]) return;
  const long long o = 3ll * vid[i];
  verts[o] = pos[3ll * i];
  verts[o + 1] = pos[3ll * i + 1];
  verts[o + 2] = pos[3ll * i + 2];
}

__global__ void __launch_bounds__(256) weld_write_tris_kernel(const int* __restrict__ ids, const int* __restrict__ keep,
                                                              const int* __restrict__ toff, int nf, int32_t* __restrict__ tris) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nf || !keep[t]) return;
  const long long o = 3ll * toff[t];
  tris[o] = ids[3ll * t];
  tris[o + 1] = ids[3ll * t + 1];
  tris[o + 2] = ids[3ll * t + 2];
}

inline int blocks_for(long long n) { return static_cast<int>((n + 255) / 256); }

// the fixed-stride triangle layout of a binary PLY, or false (host loader)
bool ply_layout(const PlyHeader& h, size_t n_bytes, PlyLayout* L) {
  if (h.format == kAscii || h.vertex < 0 || h.face < 0) return false;
  *L = PlyLayout{};
  L->big = h.format == kBinBE ? 1 : 0;
  long long off = static_cast<long long>(h.body);
  for (size_t i = 0; i < h.elems.size(); ++i) {
    const PlyElement& e = h.elems[i];
    if (static_cast<int>(i) == h.face) {
      if (e.props.size() != 1) return false;
      L->cnt_type = e.props[0].count_type;
      L->idx_type = e.props[0].type;
      L->cnt_size = type_size(L->cnt_type);
      L->idx_size = type_size(L->idx_type);
      L->f_stride = L->cnt_size + 3 * L->idx_size;
      L->f_off = off;
      L->nf = static_cast<int>(e.count);
      off += e.count * L->f_stride;
      continue;
    }
    if (!e.fixed()) return false;
    if (static_cast<int>(i) == h.vertex) {
      L->v_off = off;
      L->v_stride = e.stride();
      L->nv = static_cast<int>(e.count);
      int o = 0;
      for (size_t j = 0; j < e.props.size(); ++j) {
        for (int c = 0; c < 3; ++c) {
          if (static_cast<int>(j) == h.xyz[c]) {
            L->xo[c] = o;
            L->xt[c] = e.props[j].type;
          }
          if (static_cast<int>(j) == h.rgb[c]) L->co[c] = o;
        }
        o += type_size(e.props[j].type);
      }
      if (!h.colors) L->co[0] = L->co[1] = L->co[2] = -1;
    }
    off += e.count * e.stride();
  }
  return off == static_cast<long long>(n_bytes) && L->nv > 0 && L->nf > 0 && 3ll * L->nv < (1ll << 31) &&
         3ll * L->nf < (1ll << 31);
}

}  // namespace
}  // namespace mvlm

using namespace mvlm;

extern "C" {

size_t mvlm_mesh_parse_workspace_bytes(size_t n_bytes, int is_stl) {
  if (!is_stl) return ply_workspace_bytes(n_bytes);
  const StlLayout L = stl_layout(n_bytes);
  return L.fits ? L.total : 0;
}

int mvlm_mesh_parse_device(const uint8_t* host, size_t n_bytes, int is_stl, const char* path, void* workspace,
                           size_t workspace_bytes, void* stream, mvlm_mesh_parse_info* info) {
  MVLM_REQUIRE(info && path && (host || n_bytes == 0), "mvlm_mesh_parse_device: null pointer");
  memset(info, 0, sizeof(*info));
  info->n_bytes = n_bytes;
  info->is_stl = is_stl ? 1 : 0;
  const size_t need = mvlm_mesh_parse_workspace_bytes(n_bytes, is_stl);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  if (!is_stl) {
    PlyHeader h;
    if (parse_ply_header(host, n_bytes, path, &h) != MVLM_OK) return MVLM_E_INVALID;  // the host loader's header errors
    PlyLayout L;
    if (!ply_layout(h, n_bytes, &L)) {
      info->fallback = 1;
      return MVLM_OK;
    }
    MVLM_REQUIRE(ws && workspace_bytes >= need, "mvlm_mesh_parse_device: workspace of %zu bytes, %zu needed",
                 workspace_bytes, need);
    MVLM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mvlm_mesh_parse_device: workspace must be 256-byte aligned");
    DevHdr* hdr = reinterpret_cast<DevHdr*>(ws + round256(n_bytes));
    MVLM_CHECK_CUDA(cudaMemcpyAsync(ws, host, n_bytes, cudaMemcpyHostToDevice, s));
    MVLM_CHECK_CUDA(cudaMemsetAsync(hdr, 0, sizeof(DevHdr), s));
    ply_check_kernel<<<blocks_for(L.nf), 256, 0, s>>>(ws, L, hdr);
    count_launch(1);
    MVLM_CHECK_CUDA(cudaGetLastError());
    int fallback = 0;
    MVLM_CHECK_CUDA(cudaMemcpyAsync(&fallback, &hdr->fallback, sizeof(int), cudaMemcpyDeviceToHost, s));
    MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
    info->fallback = fallback;
    info->n_verts = L.nv;
    info->n_tris = L.nf;
    info->has_colors = h.colors ? 1 : 0;
    return MVLM_OK;
  }
  uint32_t nf_hdr = 0;
  const StlLayout L = stl_layout(n_bytes);
  if (!L.fits || !stl_is_binary(host, n_bytes, &nf_hdr)) {  // ASCII, or beyond the capacity
    info->fallback = 1;
    return MVLM_OK;
  }
  MVLM_REQUIRE(ws && workspace_bytes >= L.total, "mvlm_mesh_parse_device: workspace of %zu bytes, %zu needed",
               workspace_bytes, L.total);
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mvlm_mesh_parse_device: workspace must be 256-byte aligned");
  DevHdr* hdr = reinterpret_cast<DevHdr*>(ws + L.hdr);
  float* pos = reinterpret_cast<float*>(ws + L.pos);
  int* table = reinterpret_cast<int*>(ws + L.table);
  int* leader = reinterpret_cast<int*>(ws + L.leader);
  int* first = reinterpret_cast<int*>(ws + L.first);
  int* vid = reinterpret_cast<int*>(ws + L.vid);
  int* ids = reinterpret_cast<int*>(ws + L.ids);
  int* keep = reinterpret_cast<int*>(ws + L.keep);
  int* toff = reinterpret_cast<int*>(ws + L.toff);
  int* block_sums = reinterpret_cast<int*>(ws + L.block_sums);
  const unsigned int mask = static_cast<unsigned int>(L.slots - 1);
  MVLM_CHECK_CUDA(cudaMemcpyAsync(ws, host, n_bytes, cudaMemcpyHostToDevice, s));
  MVLM_CHECK_CUDA(cudaMemsetAsync(hdr, 0, sizeof(DevHdr), s));
  MVLM_CHECK_CUDA(cudaMemsetAsync(table, 0xff, L.slots * 4, s));
  MVLM_CHECK_CUDA(cudaMemsetAsync(first, 0, static_cast<size_t>(L.n_pad) * 4, s));  // scan padding
  MVLM_CHECK_CUDA(cudaMemsetAsync(keep, 0, static_cast<size_t>(L.f_pad) * 4, s));
  stl_decode_kernel<<<blocks_for(L.nf), 256, 0, s>>>(ws, L.nf, pos);
  weld_insert_kernel<<<blocks_for(L.n), 256, 0, s>>>(pos, L.n, table, mask);
  weld_leader_kernel<<<blocks_for(L.n), 256, 0, s>>>(pos, L.n, table, mask, leader, first);
  exclusive_scan(first, L.n_pad, block_sums, vid, &hdr->n_verts, s);
  weld_facet_kernel<<<blocks_for(L.nf), 256, 0, s>>>(leader, vid, L.nf, ids, keep);
  exclusive_scan(keep, L.f_pad, block_sums, toff, &hdr->n_tris, s);
  count_launch(10);
  MVLM_CHECK_CUDA(cudaGetLastError());
  DevHdr hh;
  MVLM_CHECK_CUDA(cudaMemcpyAsync(&hh, hdr, sizeof(hh), cudaMemcpyDeviceToHost, s));
  MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
  MVLM_REQUIRE(hh.n_tris > 0, "File %s does not contain any points.", path);
  info->n_verts = hh.n_verts;
  info->n_tris = hh.n_tris;
  return MVLM_OK;
}

int mvlm_mesh_parse_write(const mvlm_mesh_parse_info* info, const void* workspace, float* verts, uint8_t* colors,
                          int32_t* tris, void* stream) {
  MVLM_REQUIRE(info && workspace && verts && tris, "mvlm_mesh_parse_write: null pointer");
  MVLM_REQUIRE(!info->fallback && info->n_verts > 0 && info->n_tris > 0, "mvlm_mesh_parse_write: no decode to write");
  MVLM_REQUIRE(!info->has_colors || colors, "mvlm_mesh_parse_write: null colors");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint8_t* ws = static_cast<const uint8_t*>(workspace);
  if (!info->is_stl) {
    const DevHdr* hdr = reinterpret_cast<const DevHdr*>(ws + round256(info->n_bytes));
    ply_vertex_kernel<<<blocks_for(info->n_verts), 256, 0, s>>>(ws, hdr, verts, info->has_colors ? colors : nullptr);
    ply_face_kernel<<<blocks_for(info->n_tris), 256, 0, s>>>(ws, hdr, tris);
  } else {
    const StlLayout L = stl_layout(info->n_bytes);
    const float* pos = reinterpret_cast<const float*>(ws + L.pos);
    const int* first = reinterpret_cast<const int*>(ws + L.first);
    const int* vid = reinterpret_cast<const int*>(ws + L.vid);
    weld_write_verts_kernel<<<blocks_for(L.n), 256, 0, s>>>(pos, first, vid, L.n, verts);
    weld_write_tris_kernel<<<blocks_for(L.nf), 256, 0, s>>>(reinterpret_cast<const int*>(ws + L.ids),
                                                            reinterpret_cast<const int*>(ws + L.keep),
                                                            reinterpret_cast<const int*>(ws + L.toff), L.nf, tris);
  }
  count_launch(2);
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

}  // extern "C"
