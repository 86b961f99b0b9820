// Wavefront OBJ scan parser on the GPU (opt-in alternative to the host loader obj_loader.cu).
//
// Accepts exactly the language of obj_loader.cu (parse_chunk / mvlm_obj_load are the specification) and returns the
// same arrays bit for bit, with the same errors in the same order of precedence.  The host then only reads the file;
// the text crosses PCIe instead of the parsed arrays and the parse itself is a few memory-bound passes:
//
//   count  one thread per 32-byte item of the file walks the lines that START in its item (a line may run past the
//          item's end): counts its `v` lines, `vt` lines and the triangles of its faces (fan triangulation of the
//          corners; faces of fewer than 3 corners give none), flags malformed faces
//   scan   three exclusive scans of those counts (scan.cuh): the first position / uv / triangle of every item, which
//          are also the "lines seen before" that negative indices are relative to
//   parse  the same walk again: numbers of `v` / `vt` lines converted like std::from_chars(double) followed by the
//          cast to float, face corners resolved into the host's keys position << 32 | (uv + 1) in file order;
//          the first out-of-range corner (in triangulated order, like the host) by an atomic minimum of its ordinal
//   dedup  only when some corner has a uv: histogram of the corners by position, scan, scatter of their uv keys
//          into per-position buckets, per-bucket insertion sort + unique (deterministic), scan of the unique counts
//   write  (phase 2) output vertices = unique (position, uv) pairs in ascending order, and each corner's vertex
//
// Materials (MVLM_OBJ_MATERIALS, DESIGN.md 7g): the count pass also counts the `usemtl` lines and the name lines
// (`usemtl` + `mtllib`) that start in every item, two more exclusive scans give each item its first `usemtl` ordinal
// and its first name-line slot, and the parse pass stores every triangle's ordinal (the item's base plus the `usemtl`
// lines it has walked, minus one: -1 before the first) and every name line's (offset, kind, triangles before it).  The
// name lines come back to the host with the output sizes; the host reads the names from its copy of the file, maps
// each `usemtl` ordinal to a texture page and mvlm_obj_parse_tri_page writes the page of every triangle.  A file with
// more than MVLM_OBJ_MAX_NAME_LINES name lines takes the host fallback.
//
// Numbers: a token of at most 19 significant digits is converted exactly: Clinger's fast path (mantissa <= 2^53,
// |exp10| <= 22; one correctly rounded multiply or divide) or Eisel-Lemire with 128-bit products over a table of
// powers of five (the algorithm of fast_float, which libstdc++'s from_chars uses).  A token of more digits, and the
// one product Eisel-Lemire cannot round alone, set the per-file fallback flag instead: the caller re-parses such a
// file on the host, so the result is still the host's.  So does a file that exceeds the scan capacity (512 MB of
// text, 16.7M positions) or a position referenced with more than kMaxBucket corners.
//
// The per-line code is __host__ __device__: mvlm_debug_obj_parse_lines runs it serially on the CPU so that the tests
// compare it with the host parser without a GPU.
#include <climits>
#include <cstring>

#include "../../include/mvlm_b200.h"
#include "common.cuh"
#include "obj_pow5.cuh"
#include "scan.cuh"

#define HD __host__ __device__ __forceinline__

namespace mvlm {
namespace {

constexpr int kItemBytes = 32;    // bytes of the file per thread of the count / parse passes
constexpr int kMaxBucket = 1024;  // corners of one position the per-bucket insertion sort takes (else host fallback)

enum { kOk = 0, kBad = 1, kFallback = 2 };
enum { kOther = 0, kV = 1, kVT = 2, kF = 3, kUsemtl = 4, kMtllib = 5 };
constexpr int kInlineNames = 64;  // name lines copied back in the same synchronisation as the sizes

#define MVLM_POW10_TABLE                                                                                                \
  1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, \
      1e21, 1e22

__device__ const double kPow10Dev[23] = {MVLM_POW10_TABLE};
__device__ const uint64_t kPow5Dev[651 * 2] = {MVLM_POW5_128_TABLE};
#ifndef __CUDA_ARCH__
const double kPow10Host[23] = {MVLM_POW10_TABLE};
const uint64_t kPow5Host[651 * 2] = {MVLM_POW5_128_TABLE};
#endif

HD double pow10_exact(int i) {
#ifdef __CUDA_ARCH__
  return kPow10Dev[i];
#else
  return kPow10Host[i];
#endif
}

HD void pow5_128(int q, uint64_t* hi, uint64_t* lo) {
  const int i = 2 * (q + 342);
#ifdef __CUDA_ARCH__
  *hi = kPow5Dev[i];
  *lo = kPow5Dev[i + 1];
#else
  *hi = kPow5Host[i];
  *lo = kPow5Host[i + 1];
#endif
}

HD uint64_t mul_hi(uint64_t a, uint64_t b) {
#ifdef __CUDA_ARCH__
  return __umul64hi(a, b);
#else
  return static_cast<uint64_t>((static_cast<unsigned __int128>(a) * b) >> 64);
#endif
}

HD int clz64(uint64_t x) {
#ifdef __CUDA_ARCH__
  return __clzll(static_cast<long long>(x));
#else
  return __builtin_clzll(x);
#endif
}

// the fast path's one operation, never contracted with anything else
HD double mul_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __dmul_rn(a, b);
#else
  return a * b;
#endif
}
HD double div_rn(double a, double b) {
#ifdef __CUDA_ARCH__
  return __ddiv_rn(a, b);
#else
  return a / b;
#endif
}

HD double bits_double(uint64_t u) {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(static_cast<long long>(u));
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

HD uint64_t double_bits(double d) {
#ifdef __CUDA_ARCH__
  return static_cast<uint64_t>(__double_as_longlong(d));
#else
  uint64_t u;
  memcpy(&u, &d, 8);
  return u;
#endif
}

// (float)d like the host's static_cast: round to nearest even; NaN keeps its sign and becomes the quiet NaN
HD float to_float(double d) {
  if (d != d) {
    const uint32_t sign = (double_bits(d) >> 63) ? 0x80000000u : 0u;
#ifdef __CUDA_ARCH__
    return __uint_as_float(0x7fc00000u | sign);
#else
    const uint32_t u = 0x7fc00000u | sign;
    float f;
    memcpy(&f, &u, 4);
    return f;
#endif
  }
#ifdef __CUDA_ARCH__
  return __double2float_rn(d);
#else
  return static_cast<float>(d);
#endif
}

HD bool is_digit(char c) { return c >= '0' && c <= '9'; }
HD bool is_ws(char c) { return c == ' ' || c == '\t' || c == '\r'; }
HD char lower(char c) { return (c >= 'A' && c <= 'Z') ? static_cast<char>(c - 'A' + 'a') : c; }

HD bool match_ci(const char* p, const char* end, const char* word, int len) {
  if (end - p < len) return false;
  for (int i = 0; i < len; ++i)
    if (lower(p[i]) != word[i]) return false;
  return true;
}

// from_chars(double) on a token that is not a decimal number: [-]nan[(n-char-seq)], [-]inf, [-]infinity (any case)
HD int parse_infnan(const char*& p, const char* end, double* out) {
  const char* q = p;
  bool neg = false;
  if (q < end && *q == '-') {
    neg = true;
    ++q;
  }
  if (match_ci(q, end, "nan", 3)) {
    q += 3;
    if (q < end && *q == '(') {
      for (const char* r = q + 1; r < end; ++r) {
        if (*r == ')') {
          q = r + 1;
          break;
        }
        const char c = *r;
        if (!((c >= 'a' && c <= 'z') || (c >= 'A' && c <= 'Z') || is_digit(c) || c == '_')) break;
      }
    }
    *out = bits_double(0x7ff8000000000000ull | (neg ? 0x8000000000000000ull : 0ull));
    p = q;
    return kOk;
  }
  if (match_ci(q, end, "inf", 3)) {
    q += match_ci(q + 3, end, "inity", 5) ? 8 : 3;
    *out = bits_double(0x7ff0000000000000ull | (neg ? 0x8000000000000000ull : 0ull));
    p = q;
    return kOk;
  }
  return kBad;
}

// Eisel-Lemire: w * 10^q (w != 0, q in [-342, 308]) correctly rounded to binary64 bits (without the sign);
// returns kFallback for the one case the 128-bit product cannot decide (fast_float hands it to a big-number path)
HD int eisel_lemire(uint64_t w, int q, uint64_t* bits) {
  const int lz = clz64(w);
  w <<= lz;
  uint64_t p_hi, p_lo;
  pow5_128(q, &p_hi, &p_lo);
  uint64_t lo = w * p_hi, hi = mul_hi(w, p_hi);
  const uint64_t mask = 0xFFFFFFFFFFFFFFFFull >> 55;  // 52 explicit bits + 3
  if ((hi & mask) == mask) {
    const uint64_t lo2_hi = mul_hi(w, p_lo);
    lo += lo2_hi;
    if (lo2_hi > lo) ++hi;
  }
  if (lo == 0xFFFFFFFFFFFFFFFFull && !(q >= -27 && q <= 55)) return kFallback;
  const int upper = static_cast<int>(hi >> 63);
  uint64_t m = hi >> (upper + 64 - 52 - 3);
  int p2 = ((((152170 + 65536) * q) >> 16) + 63) + upper - lz + 1023;
  if (p2 <= 0) {  // subnormal (or zero)
    if (-p2 + 1 >= 64) {
      *bits = 0;
      return kOk;
    }
    m >>= -p2 + 1;
    m += (m & 1);
    m >>= 1;
    p2 = (m < (1ull << 52)) ? 0 : 1;
    *bits = (m & ((1ull << 52) - 1)) | (static_cast<uint64_t>(p2) << 52);
    return kOk;
  }
  if (lo <= 1 && q >= -4 && q <= 23 && (m & 3) == 1) {  // exactly halfway: round to even
    if ((m << (upper + 64 - 52 - 3)) == hi) m &= ~1ull;
  }
  m += (m & 1);
  m >>= 1;
  if (m >= (2ull << 52)) {
    m = 1ull << 52;
    ++p2;
  }
  m &= ~(1ull << 52);
  if (p2 >= 0x7FF) {
    *bits = 0x7FFull << 52;
    return kOk;
  }
  *bits = m | (static_cast<uint64_t>(p2) << 52);
  return kOk;
}

// std::from_chars(p, end, double) (chars_format::general, libstdc++ / fast_float semantics): kOk and p past the
// number, kBad for invalid_argument and result_out_of_range, kFallback for more than 19 significant digits
HD int from_chars_double(const char*& p, const char* end, double* out) {
  if (p >= end) return kBad;
  const char* q = p;
  const bool neg = *q == '-';
  if (neg) {
    ++q;
    if (q >= end) return kBad;
    if (!is_digit(*q) && *q != '.') return parse_infnan(p, end, out);
  }
  const char* start_digits = q;
  uint64_t w = 0;
  while (q < end && is_digit(*q)) {
    w = 10 * w + static_cast<uint64_t>(*q - '0');
    ++q;
  }
  long long digit_count = q - start_digits;
  long long exponent = 0;
  if (q < end && *q == '.') {
    ++q;
    const char* before = q;
    while (q < end && is_digit(*q)) {
      w = 10 * w + static_cast<uint64_t>(*q - '0');
      ++q;
    }
    exponent = before - q;
    digit_count -= exponent;
  }
  if (digit_count == 0) return parse_infnan(p, end, out);
  if (q < end && (*q == 'e' || *q == 'E')) {
    const char* at_e = q;
    ++q;
    bool neg_exp = false;
    if (q < end && *q == '-') {
      neg_exp = true;
      ++q;
    } else if (q < end && *q == '+') {
      ++q;
    }
    if (q >= end || !is_digit(*q)) {
      q = at_e;
    } else {
      long long e = 0;
      while (q < end && is_digit(*q)) {
        if (e < 0x10000000) e = 10 * e + (*q - '0');
        ++q;
      }
      exponent += neg_exp ? -e : e;
    }
  }
  if (digit_count > 19) {  // leading zeros (and the point) are not significant
    for (const char* s = start_digits; s < end && (*s == '0' || *s == '.'); ++s)
      if (*s == '0') --digit_count;
    if (digit_count > 19) return kFallback;
  }
  double v;
  if (exponent >= -22 && exponent <= 22 && w <= (1ull << 53)) {  // Clinger: both operands exact, one rounding
    v = static_cast<double>(w);
    v = exponent < 0 ? div_rn(v, pow10_exact(static_cast<int>(-exponent))) : mul_rn(v, pow10_exact(static_cast<int>(exponent)));
  } else {
    uint64_t bits;
    if (w == 0 || exponent < -342) {
      bits = 0;
    } else if (exponent > 308) {
      bits = 0x7FFull << 52;
    } else if (eisel_lemire(w, static_cast<int>(exponent), &bits) != kOk) {
      return kFallback;
    }
    if (w != 0 && (bits == 0 || bits == (0x7FFull << 52))) return kBad;  // result_out_of_range
    v = bits_double(bits);
  }
  *out = neg ? -v : v;
  p = q;
  return kOk;
}

// host_text.cuh parse_double: whitespace, one optional '+', from_chars
HD int parse_double(const char*& p, const char* end, double* out) {
  while (p < end && is_ws(*p)) ++p;
  if (p < end && *p == '+') ++p;
  return from_chars_double(p, end, out);
}

// std::from_chars(p, end, long long), base 10: optional '-', digits; no digits or overflow -> false
HD bool parse_int(const char*& p, const char* end, long long* out) {
  const char* q = p;
  const bool neg = q < end && *q == '-';
  if (neg) ++q;
  if (q >= end || !is_digit(*q)) return false;
  const uint64_t limit = neg ? (1ull << 63) : (1ull << 63) - 1;
  uint64_t v = 0;
  bool over = false;
  for (; q < end && is_digit(*q); ++q) {
    const uint64_t d = static_cast<uint64_t>(*q - '0');
    if (v > (limit - d) / 10) over = true;
    else v = 10 * v + d;
  }
  if (over) return false;
  *out = neg ? static_cast<long long>(0ull - v) : static_cast<long long>(v);
  p = q;
  return true;
}

HD int line_kind(const char* p, const char* eol) {
  if (eol - p >= 2 && p[0] == 'v' && p[1] == ' ') return kV;
  if (eol - p >= 3 && p[0] == 'v' && p[1] == 't' && p[2] == ' ') return kVT;
  if (eol - p >= 2 && p[0] == 'f' && p[1] == ' ') return kF;
  return kOther;
}

HD bool is_statement(const char* p, const char* eol, const char* word) {  // obj_loader.cu is_statement, 6 letters
  if (eol - p <= 6 || !(p[6] == ' ' || p[6] == '\t')) return false;
  for (int i = 0; i < 6; ++i)
    if (p[i] != word[i]) return false;
  return true;
}

// kUsemtl / kMtllib for a name line, else kOther (only asked for lines line_kind calls kOther)
HD int name_kind(const char* p, const char* eol) {
  if (is_statement(p, eol, "usemtl")) return kUsemtl;
  if (is_statement(p, eol, "mtllib")) return kMtllib;
  return kOther;
}

// the first k numbers of a `v` (k = 3, from p + 2) or `vt` (k = 2, from p + 3) line
HD int parse_numbers(const char* q, const char* eol, int k, float* out) {
  for (int i = 0; i < k; ++i) {
    double d;
    const int st = parse_double(q, eol, &d);
    if (st != kOk) return st;
    out[i] = to_float(d);
  }
  return kOk;
}

// corners of an `f` line, in order: corner(a, b) with b = 0 when the corner has no uv (OBJ indices are never 0)
template <class F>
HD int parse_face(const char* p, const char* eol, F&& corner) {
  const char* q = p + 2;
  while (true) {
    while (q < eol && is_ws(*q)) ++q;
    if (q >= eol) break;
    long long a = 0, b = 0;
    if (!parse_int(q, eol, &a)) return kBad;
    bool has_t = false;
    if (q < eol && *q == '/') {
      ++q;
      if (q < eol && *q != '/' && !is_ws(*q)) {
        if (!parse_int(q, eol, &b)) return kBad;
        has_t = true;
      }
      if (q < eol && *q == '/') {  // normal index: ignored, and so is a failure to read it
        ++q;
        long long n;
        if (q < eol && !is_ws(*q)) parse_int(q, eol, &n);
      }
    }
    corner(a, has_t ? b : 0);
  }
  return kOk;
}

// fan triangulation of a face: tri(j, a, b) for the 3 corners of every triangle (0, k, k + 1) in order
template <class T>
HD int parse_face_triangles(const char* p, const char* eol, T&& tri) {
  long long a0 = 0, b0 = 0, ap = 0, bp = 0;
  int k = 0;
  return parse_face(p, eol, [&](long long a, long long b) {
    if (k == 0) {
      a0 = a;
      b0 = b;
    } else if (k >= 2) {
      tri(0, a0, b0);
      tri(1, ap, bp);
      tri(2, a, b);
    }
    ap = a;
    bp = b;
    ++k;
  });
}

// 0 ok, 1 vertex index out of range, 2 vt index out of range (the host's checks, in its order)
HD int resolve_corner(long long a, long long b, long long v_seen, long long vt_seen, long long n_pos, long long n_tex,
                      unsigned long long* key) {
  const long long vi = a > 0 ? a - 1 : v_seen + a;
  long long ti = -1;
  if (b != 0) ti = b > 0 ? b - 1 : vt_seen + b;
  if (!(vi >= 0 && vi < n_pos)) return 1;
  if (!(ti >= -1 && ti < n_tex)) return 2;
  *key = (static_cast<unsigned long long>(vi) << 32) | static_cast<unsigned long long>(ti + 1);
  return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// Device passes
// ------------------------------------------------------------------------------------------------------------------
struct ParseHdr {
  int n_pos, n_tex, n_tri;  // totals of the three scans
  int n_corners_dedup;      // total of the histogram scan
  int n_out;                // total of the unique-count scan
  int bad, fallback, any_uv;
  int n_usemtl, n_names;    // totals of the two material scans
  unsigned int err_ord;     // first out-of-range corner (triangulated order); 0xffffffff: none
  int err_kind;             // 1 vertex, 2 vt
  long long err_a, err_b;
};

struct Layout {
  bool fits;
  int items, items_pad, p_cap, t_cap, tri_cap, p_pad;
  size_t hdr, cnt_v, cnt_vt, cnt_tri, off_v, off_vt, off_tri, block_sums, pos, tex, keys, hist, bstart, ucnt, ustart,
      bucket, total;
  // MVLM_OBJ_MATERIALS only, after everything else (the arrays above keep their offsets)
  size_t cnt_mat, cnt_name, off_mat, off_name, names, line_page, tri_ord;
};

Layout layout(size_t n, bool materials = false) {
  Layout L{};
  const size_t items = (n + kItemBytes - 1) / kItemBytes;
  const size_t items_pad = (items + kScanItems) / kScanItems * kScanItems;  // at least one block, room for a sentinel
  const size_t p_cap = n / 7 + 2, t_cap = n / 6 + 2, tri_cap = n / 2 + 2;  // "v 1-2-3", "vt 1-2", one triangle / 2 B
  const size_t p_pad = (p_cap + kScanItems) / kScanItems * kScanItems;
  L.fits = items_pad <= static_cast<size_t>(kScanItems) * kScanMaxBlocks && 3 * tri_cap < (1ull << 31);
  if (!L.fits) return L;
  L.items = static_cast<int>(items);
  L.items_pad = static_cast<int>(items_pad);
  L.p_cap = static_cast<int>(p_cap);
  L.t_cap = static_cast<int>(t_cap);
  L.tri_cap = static_cast<int>(tri_cap);
  L.p_pad = static_cast<int>(p_pad);
  size_t o = 0;
  auto take = [&](size_t bytes) {
    const size_t at = o;
    o += (bytes + 255) / 256 * 256;
    return at;
  };
  L.hdr = take(sizeof(ParseHdr));
  L.cnt_v = take(items_pad * 4);  // the three count arrays are contiguous (one memset)
  L.cnt_vt = take(items_pad * 4);
  L.cnt_tri = take(items_pad * 4);
  L.off_v = take(items_pad * 4);
  L.off_vt = take(items_pad * 4);
  L.off_tri = take(items_pad * 4);
  L.block_sums = take(kScanMaxBlocks * 4);
  L.pos = take(p_cap * 12);
  L.tex = take(t_cap * 8);
  L.keys = take(tri_cap * 3 * 8);
  L.hist = take(p_pad * 4);
  L.bstart = take(p_pad * 4);
  L.ucnt = take(p_pad * 4);
  L.ustart = take(p_pad * 4);
  L.bucket = take(tri_cap * 3 * 4);
  if (materials) {
    L.cnt_mat = take(items_pad * 4);  // contiguous with cnt_name (one memset)
    L.cnt_name = take(items_pad * 4);
    L.off_mat = take(items_pad * 4);
    L.off_name = take(items_pad * 4);
    L.names = take(static_cast<size_t>(MVLM_OBJ_MAX_NAME_LINES) * sizeof(mvlm_obj_name_line));
    L.line_page = take(static_cast<size_t>(MVLM_OBJ_MAX_NAME_LINES) * 4);
    L.tri_ord = take(tri_cap * 4);
  }
  L.total = o;
  return L;
}

// first line start in [lo, hi): lo itself if the byte before it ends a line, else the byte after the first newline
__device__ __forceinline__ long long first_line_start(const char* text, long long lo, long long hi) {
  if (lo == 0 || text[lo - 1] == '\n') return lo;
  for (long long i = lo; i < hi; ++i)
    if (text[i] == '\n') return i + 1;
  return hi;
}

__device__ __forceinline__ long long find_eol(const char* text, long long s, long long n) {
  while (s < n && text[s] != '\n') ++s;
  return s;
}

__global__ void __launch_bounds__(256) obj_count_kernel(const char* __restrict__ text, long long n, int items,
                                                        int* __restrict__ cnt_v, int* __restrict__ cnt_vt,
                                                        int* __restrict__ cnt_tri, int* __restrict__ cnt_mat,
                                                        int* __restrict__ cnt_name, ParseHdr* __restrict__ hdr) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= items) return;
  const long long lo = static_cast<long long>(c) * kItemBytes, hi = min(n, lo + kItemBytes);
  int nv = 0, nvt = 0, ntri = 0, nmat = 0, nname = 0;
  bool bad = false;
  for (long long s = first_line_start(text, lo, hi); s < hi;) {
    const long long eol = find_eol(text, s, n);
    const int kind = line_kind(text + s, text + eol);
    if (kind == kV) {
      ++nv;
    } else if (kind == kVT) {
      ++nvt;
    } else if (kind == kF) {
      int k = 0;
      if (parse_face(text + s, text + eol, [&](long long, long long) { ++k; }) != kOk) bad = true;
      ntri += k > 2 ? k - 2 : 0;
    } else if (cnt_name) {
      const int nk = name_kind(text + s, text + eol);
      nmat += nk == kUsemtl;
      nname += nk != kOther;
    }
    s = eol + 1;
  }
  cnt_v[c] = nv;
  cnt_vt[c] = nvt;
  cnt_tri[c] = ntri;
  if (cnt_name) {
    cnt_mat[c] = nmat;
    cnt_name[c] = nname;
  }
  if (bad) atomicOr(&hdr->bad, 1);
}

// kReport: the pass again after an out-of-range corner was found; only the corner of ordinal hdr->err_ord records what
// the host's message prints
template <bool kReport>
__global__ void __launch_bounds__(256) obj_parse_kernel(const char* __restrict__ text, long long n, int items,
                                                        const int* __restrict__ off_v, const int* __restrict__ off_vt,
                                                        const int* __restrict__ off_tri, ParseHdr* __restrict__ hdr,
                                                        int p_cap, int t_cap, unsigned int key_cap,
                                                        float* __restrict__ pos, float* __restrict__ tex,
                                                        unsigned long long* __restrict__ keys,
                                                        const int* __restrict__ off_mat, const int* __restrict__ off_name,
                                                        mvlm_obj_name_line* __restrict__ names,
                                                        int32_t* __restrict__ tri_ord) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= items) return;
  const long long lo = static_cast<long long>(c) * kItemBytes, hi = min(n, lo + kItemBytes);
  int vi = off_v[c], ti = off_vt[c];
  unsigned int ord = 3u * static_cast<unsigned int>(off_tri[c]);
  const long long n_pos = hdr->n_pos, n_tex = hdr->n_tex;
  const unsigned int err_ord = kReport ? hdr->err_ord : 0u;
  const bool materials = !kReport && names != nullptr;
  int mat = materials ? off_mat[c] - 1 : -1;  // ordinal of the last `usemtl` line before the current line
  int name = materials ? off_name[c] : 0;
  int bad = 0, fallback = 0, any_uv = 0;
  for (long long s = first_line_start(text, lo, hi); s < hi;) {
    const long long eol = find_eol(text, s, n);
    const char* p = text + s;
    const char* e = text + eol;
    const int kind = line_kind(p, e);
    if (!kReport && (kind == kV || kind == kVT)) {
      const bool is_v = kind == kV;
      float x[3];
      const int st = parse_numbers(p + (is_v ? 2 : 3), e, is_v ? 3 : 2, x);
      if (st == kBad) bad = 1;
      else if (st == kFallback) fallback = 1;
      else if (is_v && vi < p_cap) { pos[3ll * vi] = x[0]; pos[3ll * vi + 1] = x[1]; pos[3ll * vi + 2] = x[2]; }
      else if (!is_v && ti < t_cap) { tex[2ll * ti] = x[0]; tex[2ll * ti + 1] = x[1]; }
      else fallback = 1;
    } else if (kind == kF) {
      const long long v_seen = vi, vt_seen = ti;
      parse_face_triangles(p, e, [&](int j, long long a, long long b) {
        if (materials && j == 0 && ord < key_cap) tri_ord[ord / 3] = mat;
        unsigned long long key = 0;
        const int r = resolve_corner(a, b, v_seen, vt_seen, n_pos, n_tex, &key);
        if (kReport) {
          if (ord == err_ord) {
            hdr->err_kind = r;
            hdr->err_a = a;
            hdr->err_b = b;
          }
        } else {
          if (r != 0) atomicMin(&hdr->err_ord, ord);
          else if (static_cast<unsigned int>(key) != 0u) any_uv = 1;
          if (ord < key_cap) keys[ord] = key;
          else fallback = 1;
        }
        ++ord;
      });
    } else if (materials) {
      const int nk = name_kind(p, e);
      if (nk != kOther) {
        if (nk == kUsemtl) ++mat;
        if (name < MVLM_OBJ_MAX_NAME_LINES) {
          names[name].offset = s;
          names[name].kind = nk == kUsemtl ? 1 : 2;
          names[name].tris_before = static_cast<int32_t>(ord / 3);
        }
        ++name;
      }
    }
    if (kind == kV) ++vi;
    if (kind == kVT) ++ti;
    s = eol + 1;
  }
  if (bad) atomicOr(&hdr->bad, 1);
  if (fallback) atomicOr(&hdr->fallback, 1);
  if (any_uv) atomicOr(&hdr->any_uv, 1);
}

__global__ void __launch_bounds__(256) obj_hist_kernel(const unsigned long long* __restrict__ keys, int n_corners,
                                                       int* __restrict__ hist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_corners) atomicAdd(hist + (keys[i] >> 32), 1);
}

__global__ void __launch_bounds__(256) obj_scatter_kernel(const unsigned long long* __restrict__ keys, int n_corners,
                                                          const int* __restrict__ bstart, int* __restrict__ fill,
                                                          uint32_t* __restrict__ bucket) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_corners) return;
  const unsigned long long k = keys[i];
  const int v = static_cast<int>(k >> 32);
  bucket[bstart[v] + atomicAdd(fill + v, 1)] = static_cast<uint32_t>(k);
}

// sorts the bucket of every position in place and counts its distinct uv keys
__global__ void __launch_bounds__(256) obj_sort_unique_kernel(const int* __restrict__ bstart, int n_pos,
                                                              uint32_t* __restrict__ bucket, int* __restrict__ ucnt,
                                                              ParseHdr* __restrict__ hdr) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_pos) return;
  const int b0 = bstart[v], b1 = bstart[v + 1];
  if (b1 - b0 > kMaxBucket) {
    atomicOr(&hdr->fallback, 1);
    ucnt[v] = 0;
    return;
  }
  for (int i = b0 + 1; i < b1; ++i) {
    const uint32_t x = bucket[i];
    int j = i - 1;
    while (j >= b0 && bucket[j] > x) {
      bucket[j + 1] = bucket[j];
      --j;
    }
    bucket[j + 1] = x;
  }
  int u = 0;
  for (int i = b0; i < b1; ++i) u += (i == b0 || bucket[i] != bucket[i - 1]) ? 1 : 0;
  ucnt[v] = u;
}

__global__ void __launch_bounds__(256) obj_write_verts_kernel(const float* __restrict__ pos, const float* __restrict__ tex,
                                                              const int* __restrict__ bstart, const int* __restrict__ ustart,
                                                              const uint32_t* __restrict__ bucket, int n_pos,
                                                              float* __restrict__ verts, float* __restrict__ uvs) {
  const int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_pos) return;
  const int b0 = bstart[v], b1 = bstart[v + 1];
  long long o = ustart[v];
  for (int i = b0; i < b1; ++i) {
    if (i > b0 && bucket[i] == bucket[i - 1]) continue;
    const uint32_t t1 = bucket[i];
    verts[3 * o] = pos[3ll * v];
    verts[3 * o + 1] = pos[3ll * v + 1];
    verts[3 * o + 2] = pos[3ll * v + 2];
    uvs[2 * o] = t1 ? tex[2ll * (t1 - 1)] : 0.f;
    uvs[2 * o + 1] = t1 ? tex[2ll * (t1 - 1) + 1] : 0.f;
    ++o;
  }
}

__global__ void __launch_bounds__(256) obj_map_corners_kernel(const unsigned long long* __restrict__ keys, int n_corners,
                                                              const int* __restrict__ bstart, const int* __restrict__ ustart,
                                                              const uint32_t* __restrict__ bucket, int32_t* __restrict__ tris) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_corners) return;
  const unsigned long long k = keys[i];
  const int v = static_cast<int>(k >> 32);
  const uint32_t t1 = static_cast<uint32_t>(k);
  const int b0 = bstart[v], b1 = bstart[v + 1];
  int u = 0;
  for (int j = b0; j < b1; ++j) {  // present by construction
    if (j > b0 && bucket[j] == bucket[j - 1]) continue;
    if (bucket[j] == t1) break;
    ++u;
  }
  tris[i] = ustart[v] + u;
}

// the page of every triangle: line_page[its `usemtl` ordinal], -1 before the first `usemtl`
__global__ void __launch_bounds__(256) obj_tri_page_kernel(const int32_t* __restrict__ tri_ord, int n_tris,
                                                           const int32_t* __restrict__ line_page,
                                                           int32_t* __restrict__ tri_page) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_tris) return;
  const int m = tri_ord[i];
  tri_page[i] = m >= 0 ? line_page[m] : -1;
}

__global__ void __launch_bounds__(256) obj_positions_kernel(const unsigned long long* __restrict__ keys, int n_corners,
                                                            int32_t* __restrict__ tris) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_corners) tris[i] = static_cast<int32_t>(keys[i] >> 32);
}

inline int blocks_for(long long n) { return static_cast<int>((n + 255) / 256); }

}  // namespace
}  // namespace mvlm

using namespace mvlm;

extern "C" {

size_t mvlm_obj_parse_workspace_bytes(size_t n_bytes) { return mvlm_obj_parse_workspace_bytes_ex(n_bytes, 0); }

size_t mvlm_obj_parse_workspace_bytes_ex(size_t n_bytes, int flags) {
  const Layout L = layout(n_bytes, (flags & MVLM_OBJ_MATERIALS) != 0);
  return L.fits ? L.total : 0;
}

int mvlm_obj_parse_device(const char* text, size_t n_bytes, const char* path, void* workspace, size_t workspace_bytes,
                          void* stream, mvlm_obj_parse_info* info) {
  return mvlm_obj_parse_device_ex(text, n_bytes, path, workspace, workspace_bytes, 0, stream, info, nullptr, 0, nullptr);
}

int mvlm_obj_parse_device_ex(const char* text, size_t n_bytes, const char* path, void* workspace,
                             size_t workspace_bytes, int flags, void* stream, mvlm_obj_parse_info* info,
                             mvlm_obj_name_line* name_lines, int max_name_lines, int* n_name_lines) {
  MVLM_REQUIRE(info && path, "mvlm_obj_parse_device: null pointer");
  MVLM_REQUIRE((flags & ~MVLM_OBJ_MATERIALS) == 0, "mvlm_obj_parse_device_ex: unknown flags 0x%x", flags);
  const bool materials = (flags & MVLM_OBJ_MATERIALS) != 0;
  MVLM_REQUIRE(!materials || (name_lines && n_name_lines && max_name_lines >= MVLM_OBJ_MAX_NAME_LINES),
               "mvlm_obj_parse_device_ex: materials need a host buffer of MVLM_OBJ_MAX_NAME_LINES name lines");
  memset(info, 0, sizeof(*info));
  info->n_bytes = n_bytes;
  if (n_name_lines) *n_name_lines = 0;
  MVLM_REQUIRE(n_bytes > 0, "File %s does not contain any points.", path);
  const Layout L = layout(n_bytes, materials);
  if (!L.fits) {  // beyond the scan capacity: the host parser takes it
    info->fallback = 1;
    return MVLM_OK;
  }
  MVLM_REQUIRE(text && workspace, "mvlm_obj_parse_device: null pointer");
  MVLM_REQUIRE(workspace_bytes >= L.total, "mvlm_obj_parse_device: workspace of %zu bytes, %zu needed", workspace_bytes,
               L.total);
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 255) == 0, "mvlm_obj_parse_device: workspace must be 256-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  ParseHdr* hdr = reinterpret_cast<ParseHdr*>(ws + L.hdr);
  int* cnt_v = reinterpret_cast<int*>(ws + L.cnt_v);
  int* cnt_vt = reinterpret_cast<int*>(ws + L.cnt_vt);
  int* cnt_tri = reinterpret_cast<int*>(ws + L.cnt_tri);
  int* off_v = reinterpret_cast<int*>(ws + L.off_v);
  int* off_vt = reinterpret_cast<int*>(ws + L.off_vt);
  int* off_tri = reinterpret_cast<int*>(ws + L.off_tri);
  int* block_sums = reinterpret_cast<int*>(ws + L.block_sums);
  float* pos = reinterpret_cast<float*>(ws + L.pos);
  float* tex = reinterpret_cast<float*>(ws + L.tex);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(ws + L.keys);
  int* cnt_mat = materials ? reinterpret_cast<int*>(ws + L.cnt_mat) : nullptr;
  int* cnt_name = materials ? reinterpret_cast<int*>(ws + L.cnt_name) : nullptr;
  int* off_mat = materials ? reinterpret_cast<int*>(ws + L.off_mat) : nullptr;
  int* off_name = materials ? reinterpret_cast<int*>(ws + L.off_name) : nullptr;
  mvlm_obj_name_line* names = materials ? reinterpret_cast<mvlm_obj_name_line*>(ws + L.names) : nullptr;
  int32_t* tri_ord = materials ? reinterpret_cast<int32_t*>(ws + L.tri_ord) : nullptr;
  const long long n = static_cast<long long>(n_bytes);

  MVLM_CHECK_CUDA(cudaMemsetAsync(ws, 0, L.off_v, s));  // header + the three count arrays (padding zero)
  MVLM_CHECK_CUDA(cudaMemsetAsync(&hdr->err_ord, 0xff, sizeof(unsigned int), s));
  if (materials) MVLM_CHECK_CUDA(cudaMemsetAsync(cnt_mat, 0, L.off_mat - L.cnt_mat, s));
  obj_count_kernel<<<blocks_for(L.items), 256, 0, s>>>(text, n, L.items, cnt_v, cnt_vt, cnt_tri, cnt_mat, cnt_name, hdr);
  exclusive_scan(cnt_v, L.items_pad, block_sums, off_v, &hdr->n_pos, s);
  exclusive_scan(cnt_vt, L.items_pad, block_sums, off_vt, &hdr->n_tex, s);
  exclusive_scan(cnt_tri, L.items_pad, block_sums, off_tri, &hdr->n_tri, s);
  if (materials) {
    exclusive_scan(cnt_mat, L.items_pad, block_sums, off_mat, &hdr->n_usemtl, s);
    exclusive_scan(cnt_name, L.items_pad, block_sums, off_name, &hdr->n_names, s);
    count_launch(6);
  }
  obj_parse_kernel<false><<<blocks_for(L.items), 256, 0, s>>>(text, n, L.items, off_v, off_vt, off_tri, hdr, L.p_cap,
                                                              L.t_cap, 3u * L.tri_cap, pos, tex, keys, off_mat,
                                                              off_name, names, tri_ord);
  count_launch(11);
  MVLM_CHECK_CUDA(cudaGetLastError());
  ParseHdr h;
  MVLM_CHECK_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, s));
  if (materials)  // the first name lines travel with the sizes; a file with more takes one more copy below
    MVLM_CHECK_CUDA(cudaMemcpyAsync(name_lines, names, kInlineNames * sizeof(mvlm_obj_name_line), cudaMemcpyDeviceToHost, s));
  MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
  // the host parser's order of precedence: malformed line, no points, first out-of-range corner
  if (h.fallback) {
    info->fallback = 1;
    return MVLM_OK;
  }
  MVLM_REQUIRE(!h.bad, "mvlm_obj_load: malformed v / vt / f line in %s", path);
  MVLM_REQUIRE(h.n_pos > 0, "File %s does not contain any points.", path);
  if (h.err_ord != 0xffffffffu) {
    obj_parse_kernel<true><<<blocks_for(L.items), 256, 0, s>>>(text, n, L.items, off_v, off_vt, off_tri, hdr, L.p_cap,
                                                               L.t_cap, 3u * L.tri_cap, pos, tex, keys, nullptr,
                                                               nullptr, nullptr, nullptr);
    count_launch(1);
    MVLM_CHECK_CUDA(cudaGetLastError());
    MVLM_CHECK_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, s));
    MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
    MVLM_REQUIRE(h.err_kind != 1, "mvlm_obj_load: face references vertex %lld of %zu in %s", h.err_a,
                 static_cast<size_t>(h.n_pos), path);
    MVLM_REQUIRE(false, "mvlm_obj_load: face references vt %lld of %zu in %s", h.err_b, static_cast<size_t>(h.n_tex), path);
  }
  const int n_corners = 3 * h.n_tri;
  if (h.any_uv) {
    if (h.n_pos >= L.p_pad) {  // (cannot happen: p_cap bounds the `v` lines) -- never index past the arrays
      info->fallback = 1;
      return MVLM_OK;
    }
    int* hist = reinterpret_cast<int*>(ws + L.hist);
    int* bstart = reinterpret_cast<int*>(ws + L.bstart);
    int* ucnt = reinterpret_cast<int*>(ws + L.ucnt);
    int* ustart = reinterpret_cast<int*>(ws + L.ustart);
    uint32_t* bucket = reinterpret_cast<uint32_t*>(ws + L.bucket);
    const int p_pad = (h.n_pos + kScanItems) / kScanItems * kScanItems;
    if (p_pad > kScanItems * kScanMaxBlocks) {
      info->fallback = 1;
      return MVLM_OK;
    }
    MVLM_CHECK_CUDA(cudaMemsetAsync(hist, 0, static_cast<size_t>(p_pad) * 4, s));
    MVLM_CHECK_CUDA(cudaMemsetAsync(ucnt, 0, static_cast<size_t>(p_pad) * 4, s));
    obj_hist_kernel<<<blocks_for(n_corners), 256, 0, s>>>(keys, n_corners, hist);
    exclusive_scan(hist, p_pad, block_sums, bstart, &hdr->n_corners_dedup, s);
    MVLM_CHECK_CUDA(cudaMemsetAsync(hist, 0, static_cast<size_t>(p_pad) * 4, s));  // now the fill counters
    obj_scatter_kernel<<<blocks_for(n_corners), 256, 0, s>>>(keys, n_corners, bstart, hist, bucket);
    obj_sort_unique_kernel<<<blocks_for(h.n_pos), 256, 0, s>>>(bstart, h.n_pos, bucket, ucnt, hdr);
    exclusive_scan(ucnt, p_pad, block_sums, ustart, &hdr->n_out, s);
    count_launch(9);
    MVLM_CHECK_CUDA(cudaGetLastError());
    MVLM_CHECK_CUDA(cudaMemcpyAsync(&h, hdr, sizeof(h), cudaMemcpyDeviceToHost, s));
    MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
    if (h.fallback) {
      info->fallback = 1;
      return MVLM_OK;
    }
  }
  if (materials) {
    if (h.n_names > MVLM_OBJ_MAX_NAME_LINES) {
      info->fallback = 1;
      return MVLM_OK;
    }
    if (h.n_names > kInlineNames) {
      MVLM_CHECK_CUDA(cudaMemcpyAsync(name_lines + kInlineNames, names + kInlineNames,
                                      static_cast<size_t>(h.n_names - kInlineNames) * sizeof(mvlm_obj_name_line),
                                      cudaMemcpyDeviceToHost, s));
      MVLM_CHECK_CUDA(cudaStreamSynchronize(s));
    }
    *n_name_lines = h.n_names;
  }
  info->n_verts = h.any_uv ? h.n_out : h.n_pos;
  info->n_tris = h.n_tri;
  info->has_uv = h.any_uv ? 1 : 0;
  info->n_positions = h.n_pos;
  return MVLM_OK;
}

int mvlm_obj_parse_write(const mvlm_obj_parse_info* info, const void* workspace, float* verts, float* uvs, int32_t* tris,
                         void* stream) {
  MVLM_REQUIRE(info && workspace && verts && (tris || info->n_tris == 0), "mvlm_obj_parse_write: null pointer");
  MVLM_REQUIRE(!info->fallback && info->n_positions > 0, "mvlm_obj_parse_write: no parse to write");
  MVLM_REQUIRE(!info->has_uv || uvs, "mvlm_obj_parse_write: null uvs");
  const Layout L = layout(info->n_bytes);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const uint8_t* ws = static_cast<const uint8_t*>(workspace);
  const float* pos = reinterpret_cast<const float*>(ws + L.pos);
  const unsigned long long* keys = reinterpret_cast<const unsigned long long*>(ws + L.keys);
  const int n_corners = 3 * info->n_tris;
  if (!info->has_uv) {
    MVLM_CHECK_CUDA(cudaMemcpyAsync(verts, pos, static_cast<size_t>(info->n_positions) * 12, cudaMemcpyDeviceToDevice, s));
    if (n_corners > 0) {
      obj_positions_kernel<<<blocks_for(n_corners), 256, 0, s>>>(keys, n_corners, tris);
      count_launch(1);
    }
  } else {
    const float* tex = reinterpret_cast<const float*>(ws + L.tex);
    const int* bstart = reinterpret_cast<const int*>(ws + L.bstart);
    const int* ustart = reinterpret_cast<const int*>(ws + L.ustart);
    const uint32_t* bucket = reinterpret_cast<const uint32_t*>(ws + L.bucket);
    obj_write_verts_kernel<<<blocks_for(info->n_positions), 256, 0, s>>>(pos, tex, bstart, ustart, bucket,
                                                                        info->n_positions, verts, uvs);
    obj_map_corners_kernel<<<blocks_for(n_corners), 256, 0, s>>>(keys, n_corners, bstart, ustart, bucket, tris);
    count_launch(2);
  }
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

int mvlm_obj_parse_tri_page(const mvlm_obj_parse_info* info, void* workspace, const int32_t* line_page, int n_usemtl,
                            int32_t* tri_page, void* stream) {
  MVLM_REQUIRE(info && workspace && (line_page || n_usemtl == 0) && (tri_page || info->n_tris == 0),
               "mvlm_obj_parse_tri_page: null pointer");
  MVLM_REQUIRE(!info->fallback && info->n_positions > 0, "mvlm_obj_parse_tri_page: no parse to write");
  MVLM_REQUIRE(n_usemtl >= 0 && n_usemtl <= MVLM_OBJ_MAX_NAME_LINES, "mvlm_obj_parse_tri_page: %d usemtl lines",
               n_usemtl);
  const Layout L = layout(info->n_bytes, true);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  int32_t* table = reinterpret_cast<int32_t*>(ws + L.line_page);
  if (n_usemtl > 0)
    MVLM_CHECK_CUDA(cudaMemcpyAsync(table, line_page, static_cast<size_t>(n_usemtl) * 4, cudaMemcpyHostToDevice, s));
  if (info->n_tris > 0) {
    obj_tri_page_kernel<<<blocks_for(info->n_tris), 256, 0, s>>>(reinterpret_cast<const int32_t*>(ws + L.tri_ord),
                                                                 info->n_tris, table, tri_page);
    count_launch(1);
  }
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

int mvlm_debug_obj_parse_lines(const char* text, size_t len, int max_lines, int* n_lines, int32_t* kind, int32_t* status,
                               float* values, int32_t* n_tris, long long* corners, long long max_corners) {
  MVLM_REQUIRE((text || len == 0) && n_lines && kind && status && values && n_tris && (corners || max_corners == 0),
               "mvlm_debug_obj_parse_lines: null pointer");
  const char* end = text + len;
  long long nc = 0;
  int i = 0;
  for (const char* p = text; p < end; ++i) {
    MVLM_REQUIRE(i < max_lines, "mvlm_debug_obj_parse_lines: more than %d lines", max_lines);
    const char* eol = static_cast<const char*>(memchr(p, '\n', static_cast<size_t>(end - p)));
    if (!eol) eol = end;
    const int k = line_kind(p, eol);
    kind[i] = k;
    status[i] = kOk;
    n_tris[i] = 0;
    values[3 * i] = values[3 * i + 1] = values[3 * i + 2] = 0.f;
    if (k == kV || k == kVT) {
      status[i] = parse_numbers(p + (k == kV ? 2 : 3), eol, k == kV ? 3 : 2, values + 3 * i);
    } else if (k == kF) {
      const long long nc0 = nc;
      bool full = false;
      status[i] = parse_face_triangles(p, eol, [&](int, long long a, long long b) {
        if (nc >= max_corners) {
          full = true;
          return;
        }
        corners[2 * nc] = a;
        corners[2 * nc + 1] = b;
        ++nc;
      });
      MVLM_REQUIRE(!full, "mvlm_debug_obj_parse_lines: more than %lld corners", max_corners);
      n_tris[i] = static_cast<int32_t>((nc - nc0) / 3);
    }
    p = eol + 1;
  }
  *n_lines = i;
  return MVLM_OK;
}

}  // extern "C"
