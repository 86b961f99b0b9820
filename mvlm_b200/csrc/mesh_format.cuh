// PLY / STL scan formats: what the host loader (mesh_loader.cu) and the GPU decoder (mesh_parse.cu) share, so that the
// two read the same language and produce the same bits.
//
//   - PLY header parser (host): elements, scalar and list properties, which vertex properties are used
//   - scalar readers (host and device): one value of a PLY type at a byte address, either endianness
//   - the f64 -> f32 conversion and the weld key of a corner (host and device)
//   - the binary STL size rule
//
// The rules themselves are DESIGN.md 7f.
#pragma once

#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

#define MVLM_HD __host__ __device__ __forceinline__

namespace mvlm {
namespace mesh {

enum PlyType { kChar = 0, kUChar, kShort, kUShort, kInt, kUInt, kFloat, kDouble };
enum PlyFormat { kAscii = 0, kBinLE, kBinBE };

MVLM_HD int type_size(int t) {
  switch (t) {
    case kChar: case kUChar: return 1;
    case kShort: case kUShort: return 2;
    case kInt: case kUInt: case kFloat: return 4;
    default: return 8;
  }
}

MVLM_HD uint64_t load_le_be(const uint8_t* p, int n, bool big) {
  uint64_t v = 0;
  if (big) {
    for (int i = 0; i < n; ++i) v = (v << 8) | p[i];
  } else {
    for (int i = n - 1; i >= 0; --i) v = (v << 8) | p[i];
  }
  return v;
}

MVLM_HD float bits_to_float(uint32_t u) {
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}

MVLM_HD uint32_t float_to_bits(float f) {
#ifdef __CUDA_ARCH__
  return __float_as_uint(f);
#else
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
#endif
}

MVLM_HD double bits_to_double(uint64_t u) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(static_cast<long long>(u));
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

MVLM_HD uint64_t double_to_bits(double d) {
#ifdef __CUDA_ARCH__
  return static_cast<uint64_t>(__double_as_longlong(d));
#else
  uint64_t u;
  memcpy(&u, &d, 8);
  return u;
#endif
}

// static_cast<float>(d), round to nearest even; a NaN becomes the quiet NaN of its sign (the GPU OBJ parser's rule), so
// host and device agree on its bits too
MVLM_HD float f64_to_f32(double d) {
  if (d != d) return bits_to_float(0x7fc00000u | ((double_to_bits(d) >> 63) ? 0x80000000u : 0u));
#ifdef __CUDA_ARCH__
  return __double2float_rn(d);
#else
  return static_cast<float>(d);
#endif
}

// integer value of an integer-typed scalar
MVLM_HD long long read_int(const uint8_t* p, int t, bool big) {
  const uint64_t u = load_le_be(p, type_size(t), big);
  switch (t) {
    case kChar: return static_cast<int8_t>(u);
    case kUChar: return static_cast<uint8_t>(u);
    case kShort: return static_cast<int16_t>(u);
    case kUShort: return static_cast<uint16_t>(u);
    case kInt: return static_cast<int32_t>(u);
    default: return static_cast<uint32_t>(u);
  }
}

// a coordinate of any type as float32: float keeps its bits, double and integers are converted (round to nearest)
MVLM_HD float read_coord(const uint8_t* p, int t, bool big) {
  if (t == kFloat) return bits_to_float(static_cast<uint32_t>(load_le_be(p, 4, big)));
  if (t == kDouble) return f64_to_f32(bits_to_double(load_le_be(p, 8, big)));
  return f64_to_f32(static_cast<double>(read_int(p, t, big)));
}

// Weld key of a corner: the three coordinate bit patterns with -0.0 folded onto +0.0, so that keys are equal exactly when
// the floats compare equal.  A corner with a NaN coordinate equals nothing (not even itself) and is never merged.
MVLM_HD uint32_t weld_bits(float f) {
  const uint32_t u = float_to_bits(f);
  return u == 0x80000000u ? 0u : u;
}
MVLM_HD bool weld_is_nan(float x, float y, float z) { return x != x || y != y || z != z; }
MVLM_HD uint32_t weld_hash(uint32_t x, uint32_t y, uint32_t z) {
  uint32_t h = x * 0x9E3779B1u;
  h ^= (y + 0x7F4A7C15u) * 0x85EBCA77u;
  h ^= (z + 0x165667B1u) * 0xC2B2AE3Du;
  h ^= h >> 15;
  h *= 0x2C1B3C6Du;
  h ^= h >> 12;
  return h;
}
// open-addressing table of at least twice as many slots as keys, a power of two
inline size_t weld_table_slots(size_t n_keys) {
  size_t s = 1024;
  while (s < 2 * n_keys) s <<= 1;
  return s;
}

// Binary STL iff the size is at least 84 and equals 84 + 50 n, n = the little-endian uint32 at byte 80
inline bool stl_is_binary(const uint8_t* data, size_t n, uint32_t* n_facets) {
  if (n < 84) return false;
  const uint32_t f = static_cast<uint32_t>(load_le_be(data + 80, 4, false));
  *n_facets = f;
  return static_cast<unsigned long long>(n) == 84ull + 50ull * f;
}

struct PlyProp {
  std::string name;
  int type = kFloat;      // scalar type, or the item type of a list
  bool list = false;
  int count_type = kUChar;
};
struct PlyElement {
  std::string name;
  long long count = 0;
  std::vector<PlyProp> props;
  bool fixed() const {  // no list property: records of one size
    for (const PlyProp& p : props)
      if (p.list) return false;
    return true;
  }
  int stride() const {
    int s = 0;
    for (const PlyProp& p : props) s += type_size(p.type);
    return s;
  }
};
struct PlyHeader {
  int format = kAscii;
  size_t body = 0;                 // byte offset of the body (after the end_header line)
  std::vector<PlyElement> elems;
  int vertex = -1, face = -1;      // element indices
  int xyz[3] = {-1, -1, -1};       // property indices within the vertex element
  int rgb[3] = {-1, -1, -1};       // red green blue, used only when all three are uchar
  bool colors = false;
  int face_list = -1;              // the vertex_indices / vertex_index list within the face element
};

// Parses the header of a PLY file (host).  Errors are reported with mvlm::set_error and a nonzero return.
int parse_ply_header(const uint8_t* data, size_t n, const char* path, PlyHeader* h);

}  // namespace mesh
}  // namespace mvlm
