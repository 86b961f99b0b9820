// Native PLY / STL scan loader (host code): the specification of the two formats and the reference the GPU decoder
// (mesh_parse.cu) is checked against.  Rules: DESIGN.md 7f; the numpy restatement is tests/mesh_ref.py.
//
//   PLY  ascii, binary_little_endian, binary_big_endian.  `vertex` x y z (any numeric type -> float32), red green blue
//        as colours when all three are uchar; `face` vertex_indices / vertex_index list, fan-triangulated (0, k, k + 1)
//        like the OBJ loader; every other property and element is skipped.
//   STL  binary iff size == 84 + 50 n (n = uint32 at byte 80), else ASCII.  The triangle soup is welded: corners with
//        equal float32 coordinates (+0 == -0, NaN never) become one vertex, numbered in order of first occurrence, and
//        facets that become degenerate are dropped.
//
// ASCII bodies are split at line boundaries into one chunk per thread and each chunk is converted with std::from_chars
// (correctly rounded, like the OBJ loader) before one serial pass interprets the values.
#include <charconv>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/mvlm_b200.h"
#include "common.cuh"
#include "host_text.cuh"
#include "mesh_format.cuh"

struct mvlm_mesh {
  std::vector<float> verts;
  std::vector<uint8_t> colors;  // (Nv,3) when has_colors
  std::vector<int32_t> tris;
  bool has_colors = false;
};

namespace mvlm {
namespace mesh {

namespace {

bool type_from_name(const std::string& s, int* t) {
  static const char* names[8][2] = {{"char", "int8"},   {"uchar", "uint8"}, {"short", "int16"},  {"ushort", "uint16"},
                                    {"int", "int32"},   {"uint", "uint32"}, {"float", "float32"}, {"double", "float64"}};
  for (int i = 0; i < 8; ++i)
    if (s == names[i][0] || s == names[i][1]) {
      *t = i;
      return true;
    }
  return false;
}

std::vector<std::string> split_ws(const char* p, const char* end) {
  std::vector<std::string> out;
  while (p < end) {
    while (p < end && (*p == ' ' || *p == '\t' || *p == '\r')) ++p;
    const char* s = p;
    while (p < end && *p != ' ' && *p != '\t' && *p != '\r') ++p;
    if (p > s) out.emplace_back(s, p);
  }
  return out;
}

}  // namespace

int parse_ply_header(const uint8_t* data, size_t n, const char* path, PlyHeader* h) {
  const char* base = reinterpret_cast<const char*>(data);
  const char* end = base + n;
  const char* p = base;
  int line_no = 0;
  bool have_format = false;
  *h = PlyHeader();
  while (true) {
    MVLM_REQUIRE(p < end, "mvlm_mesh_load: malformed PLY header in %s (no end_header)", path);
    const char* eol = static_cast<const char*>(memchr(p, '\n', static_cast<size_t>(end - p)));
    MVLM_REQUIRE(eol != nullptr, "mvlm_mesh_load: malformed PLY header in %s (no end_header)", path);
    const std::vector<std::string> tok = split_ws(p, eol);
    p = eol + 1;
    if (line_no++ == 0) {
      MVLM_REQUIRE(tok.size() == 1 && tok[0] == "ply", "mvlm_mesh_load: %s is not a PLY file (no 'ply' line)", path);
      continue;
    }
    if (tok.empty()) continue;
    const std::string& k = tok[0];
    if (k == "comment" || k == "obj_info") continue;
    if (k == "end_header") break;
    if (k == "format") {
      MVLM_REQUIRE(tok.size() == 3 && tok[2] == "1.0", "mvlm_mesh_load: malformed PLY header in %s (format line)", path);
      if (tok[1] == "ascii") h->format = kAscii;
      else if (tok[1] == "binary_little_endian") h->format = kBinLE;
      else if (tok[1] == "binary_big_endian") h->format = kBinBE;
      else MVLM_REQUIRE(false, "mvlm_mesh_load: unsupported PLY format '%s' in %s", tok[1].c_str(), path);
      have_format = true;
    } else if (k == "element") {
      MVLM_REQUIRE(tok.size() == 3, "mvlm_mesh_load: malformed PLY header in %s (element line)", path);
      PlyElement e;
      e.name = tok[1];
      const char* s = tok[2].data();
      const auto r = std::from_chars(s, s + tok[2].size(), e.count);
      MVLM_REQUIRE(r.ec == std::errc() && r.ptr == s + tok[2].size() && e.count >= 0 && e.count < (1ll << 31),
                   "mvlm_mesh_load: malformed PLY header in %s (element count '%s')", path, tok[2].c_str());
      h->elems.push_back(e);
    } else if (k == "property") {
      MVLM_REQUIRE(!h->elems.empty(), "mvlm_mesh_load: malformed PLY header in %s (property before element)", path);
      PlyProp q;
      if (tok.size() == 5 && tok[1] == "list") {
        q.list = true;
        MVLM_REQUIRE(type_from_name(tok[2], &q.count_type) && type_from_name(tok[3], &q.type),
                     "mvlm_mesh_load: unsupported PLY property type in %s (list %s %s)", path, tok[2].c_str(),
                     tok[3].c_str());
        MVLM_REQUIRE(q.count_type < kFloat, "mvlm_mesh_load: unsupported PLY property type in %s (list count %s)", path,
                     tok[2].c_str());
        q.name = tok[4];
      } else {
        MVLM_REQUIRE(tok.size() == 3, "mvlm_mesh_load: malformed PLY header in %s (property line)", path);
        MVLM_REQUIRE(type_from_name(tok[1], &q.type), "mvlm_mesh_load: unsupported PLY property type '%s' in %s",
                     tok[1].c_str(), path);
        q.name = tok[2];
      }
      h->elems.back().props.push_back(q);
    } else {
      MVLM_REQUIRE(false, "mvlm_mesh_load: malformed PLY header in %s (unknown keyword '%s')", path, k.c_str());
    }
  }
  MVLM_REQUIRE(have_format, "mvlm_mesh_load: malformed PLY header in %s (no format line)", path);
  h->body = static_cast<size_t>(p - base);
  for (size_t i = 0; i < h->elems.size(); ++i) {
    const PlyElement& e = h->elems[i];
    if (e.name == "vertex" && h->vertex < 0) {
      h->vertex = static_cast<int>(i);
      static const char* xyz[3] = {"x", "y", "z"};
      static const char* rgb[3] = {"red", "green", "blue"};
      for (size_t j = 0; j < e.props.size(); ++j)
        for (int c = 0; c < 3; ++c) {
          if (!e.props[j].list && e.props[j].name == xyz[c] && h->xyz[c] < 0) h->xyz[c] = static_cast<int>(j);
          if (!e.props[j].list && e.props[j].name == rgb[c] && h->rgb[c] < 0) h->rgb[c] = static_cast<int>(j);
        }
      MVLM_REQUIRE(h->xyz[0] >= 0 && h->xyz[1] >= 0 && h->xyz[2] >= 0,
                   "mvlm_mesh_load: malformed PLY header in %s (vertex element without x y z)", path);
      h->colors = true;
      for (int c = 0; c < 3; ++c) h->colors = h->colors && h->rgb[c] >= 0 && e.props[static_cast<size_t>(h->rgb[c])].type == kUChar;
    } else if (e.name == "face" && h->face < 0) {
      h->face = static_cast<int>(i);
      for (size_t j = 0; j < e.props.size(); ++j)
        if (e.props[j].list && (e.props[j].name == "vertex_indices" || e.props[j].name == "vertex_index")) {
          MVLM_REQUIRE(h->face_list < 0, "mvlm_mesh_load: malformed PLY header in %s (two face index lists)", path);
          h->face_list = static_cast<int>(j);
        }
      MVLM_REQUIRE(h->face_list >= 0, "mvlm_mesh_load: malformed PLY header in %s (face element without vertex_indices)",
                   path);
      MVLM_REQUIRE(e.props[static_cast<size_t>(h->face_list)].type < kFloat,
                   "mvlm_mesh_load: unsupported PLY property type in %s (float face indices)", path);
    }
  }
  return MVLM_OK;
}

}  // namespace mesh

namespace {

using namespace mesh;

inline bool is_space(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n'; }

// ---- PLY body readers ------------------------------------------------------------------------------------------------
struct BinReader {
  const uint8_t* p;
  const uint8_t* end;
  bool big;
  const char* error() const { return "truncated binary PLY body"; }
  bool room(long long n, int t) const { return n <= (end - p) / type_size(t); }
  bool take(int t, const uint8_t** at) {
    const int s = type_size(t);
    if (end - p < s) return false;
    *at = p;
    p += s;
    return true;
  }
  bool integer(int t, long long* v) {  // t: an integer type (the header parser checks counts and indices)
    const uint8_t* a;
    if (!take(t, &a)) return false;
    *v = read_int(a, t, big);
    return true;
  }
  bool coord(int t, float* v) {
    const uint8_t* a;
    if (!take(t, &a)) return false;
    *v = read_coord(a, t, big);
    return true;
  }
  bool skip(int t) {
    const uint8_t* a;
    return take(t, &a);
  }
};

// every token of the body converted to double; integer-typed properties must hold an integral value in range
struct AsciiReader {
  const std::vector<double>* vals;
  size_t i = 0;
  bool bad_number = false;
  const char* error() const { return bad_number ? "malformed ASCII number in the PLY body" : "truncated PLY body"; }
  bool room(long long n, int) const { return static_cast<size_t>(n) <= vals->size() - i; }
  bool integer(int t, long long* v) {
    if (i >= vals->size()) return false;
    const double d = (*vals)[i++];
    static const double lo[6] = {-128.0, 0.0, -32768.0, 0.0, -2147483648.0, 0.0};
    static const double hi[6] = {127.0, 255.0, 32767.0, 65535.0, 2147483647.0, 4294967295.0};
    if (!(d >= lo[t] && d <= hi[t]) || d != std::floor(d)) {
      bad_number = true;
      return false;
    }
    *v = static_cast<long long>(d);
    return true;
  }
  bool coord(int t, float* v) {
    if (i >= vals->size()) return false;
    const double d = (*vals)[i++];
    if (t < kFloat && d != std::floor(d)) {
      bad_number = true;
      return false;
    }
    *v = f64_to_f32(d);
    return true;
  }
  bool skip(int) {
    if (i >= vals->size()) return false;
    ++i;
    return true;
  }
};

struct Tokens {
  std::vector<double> v;
  bool bad = false;
};

void tokenize(const char* p, const char* end, Tokens* out) {
  while (p < end) {
    while (p < end && is_space(*p)) ++p;
    if (p >= end) break;
    double d;
    const char* q = p;
    if (!parse_double(q, end, &d) || (q < end && !is_space(*q))) {
      out->bad = true;
      return;
    }
    out->v.push_back(d);
    p = q;
  }
}

template <class R>
int read_ply_body(const PlyHeader& h, R& rd, const char* path, mvlm_mesh* m) {
  const long long nv = h.vertex >= 0 ? h.elems[static_cast<size_t>(h.vertex)].count : 0;
  m->has_colors = h.colors;
  m->verts.assign(static_cast<size_t>(nv) * 3, 0.f);
  if (h.colors) m->colors.assign(static_cast<size_t>(nv) * 3, 0);
  std::vector<long long> fv;
  for (size_t ei = 0; ei < h.elems.size(); ++ei) {
    const PlyElement& e = h.elems[ei];
    const int role = static_cast<int>(ei) == h.vertex ? 1 : static_cast<int>(ei) == h.face ? 2 : 0;
    for (long long r = 0; r < e.count; ++r) {
      for (size_t pi = 0; pi < e.props.size(); ++pi) {
        const PlyProp& q = e.props[pi];
        if (q.list) {
          long long cnt;
          MVLM_REQUIRE(rd.integer(q.count_type, &cnt), "mvlm_mesh_load: %s in %s", rd.error(), path);
          MVLM_REQUIRE(cnt >= 0, "mvlm_mesh_load: negative list length in %s", path);
          MVLM_REQUIRE(rd.room(cnt, q.type), "mvlm_mesh_load: %s in %s", rd.error(), path);
          if (role == 2 && static_cast<int>(pi) == h.face_list) {
            fv.resize(static_cast<size_t>(cnt));
            for (long long j = 0; j < cnt; ++j)
              MVLM_REQUIRE(rd.integer(q.type, &fv[static_cast<size_t>(j)]), "mvlm_mesh_load: %s in %s", rd.error(), path);
            for (long long k = 1; k + 1 < cnt; ++k) {
              const long long c[3] = {fv[0], fv[static_cast<size_t>(k)], fv[static_cast<size_t>(k) + 1]};
              for (long long x : c) {
                MVLM_REQUIRE(x >= 0 && x < nv, "mvlm_mesh_load: face references vertex %lld of %lld in %s", x, nv, path);
                m->tris.push_back(static_cast<int32_t>(x));
              }
            }
          } else {
            for (long long j = 0; j < cnt; ++j) MVLM_REQUIRE(rd.skip(q.type), "mvlm_mesh_load: %s in %s", rd.error(), path);
          }
          continue;
        }
        bool ok = true;
        if (role == 1) {
          const size_t o = static_cast<size_t>(r) * 3;
          const int ip = static_cast<int>(pi);
          if (ip == h.xyz[0] || ip == h.xyz[1] || ip == h.xyz[2]) {
            float v;
            ok = rd.coord(q.type, &v);
            for (int c = 0; c < 3; ++c)
              if (ip == h.xyz[c]) m->verts[o + static_cast<size_t>(c)] = v;
          } else if (h.colors && (ip == h.rgb[0] || ip == h.rgb[1] || ip == h.rgb[2])) {
            long long v = 0;
            ok = rd.integer(q.type, &v);
            for (int c = 0; c < 3; ++c)
              if (ip == h.rgb[c]) m->colors[o + static_cast<size_t>(c)] = static_cast<uint8_t>(v);
          } else {
            ok = rd.skip(q.type);
          }
        } else {
          ok = rd.skip(q.type);
        }
        MVLM_REQUIRE(ok, "mvlm_mesh_load: %s in %s", rd.error(), path);
      }
    }
  }
  return MVLM_OK;
}

int load_ply(const std::string& buf, const char* path, int n_threads, mvlm_mesh* m) {
  const uint8_t* data = reinterpret_cast<const uint8_t*>(buf.data());
  PlyHeader h;
  if (parse_ply_header(data, buf.size(), path, &h) != MVLM_OK) return MVLM_E_INVALID;
  if (h.format == kAscii) {
    const char* b = buf.data() + h.body;
    std::vector<Tokens> chunks = parallel_chunks<Tokens>(b, buf.data() + buf.size(), n_threads, tokenize);
    Tokens all;
    for (Tokens& c : chunks) {
      MVLM_REQUIRE(!c.bad, "mvlm_mesh_load: malformed ASCII number in %s", path);
      all.v.insert(all.v.end(), c.v.begin(), c.v.end());
    }
    AsciiReader rd{&all.v};
    return read_ply_body(h, rd, path, m);
  }
  BinReader rd{data + h.body, data + buf.size(), h.format == kBinBE};
  return read_ply_body(h, rd, path, m);
}

// ---- STL -------------------------------------------------------------------------------------------------------------
// corners (3 per facet, xyz) -> m->verts (first occurrences) and m->tris (non-degenerate facets, file order)
void weld(const std::vector<float>& c, mvlm_mesh* m) {
  const size_t n = c.size() / 3;
  const size_t slots = weld_table_slots(n);
  const size_t mask = slots - 1;
  std::vector<int32_t> table(slots, -1);  // vertex id
  std::vector<int32_t> id(n);
  m->verts.clear();
  m->verts.reserve(c.size() / 4);
  for (size_t i = 0; i < n; ++i) {
    const float x = c[3 * i], y = c[3 * i + 1], z = c[3 * i + 2];
    const int32_t next = static_cast<int32_t>(m->verts.size() / 3);
    if (weld_is_nan(x, y, z)) {
      id[i] = next;
      m->verts.insert(m->verts.end(), {x, y, z});
      continue;
    }
    const uint32_t kx = weld_bits(x), ky = weld_bits(y), kz = weld_bits(z);
    for (size_t s = weld_hash(kx, ky, kz) & mask;; s = (s + 1) & mask) {
      const int32_t v = table[s];
      if (v < 0) {
        table[s] = next;
        id[i] = next;
        m->verts.insert(m->verts.end(), {x, y, z});
        break;
      }
      const float* q = &m->verts[static_cast<size_t>(v) * 3];
      if (weld_bits(q[0]) == kx && weld_bits(q[1]) == ky && weld_bits(q[2]) == kz) {
        id[i] = v;
        break;
      }
    }
  }
  m->tris.clear();
  for (size_t t = 0; t < n / 3; ++t) {
    const int32_t a = id[3 * t], b = id[3 * t + 1], d = id[3 * t + 2];
    if (a == b || b == d || a == d) continue;
    m->tris.insert(m->tris.end(), {a, b, d});
  }
}

enum { kEvFacet = 0, kEvVertex, kEvEndFacet, kEvBadLine, kEvBadNumber };
struct StlEvent {
  int kind;
  float xyz[3];
};

bool word(const char* p, const char* e, const char* w) {
  const size_t n = strlen(w);
  return static_cast<size_t>(e - p) >= n && memcmp(p, w, n) == 0 && (static_cast<size_t>(e - p) == n || is_space(p[n]));
}

void stl_lines(const char* p, const char* end, std::vector<StlEvent>* out) {
  while (p < end) {
    const char* eol = static_cast<const char*>(memchr(p, '\n', static_cast<size_t>(end - p)));
    if (!eol) eol = end;
    const char* q = p;
    while (q < eol && is_space(*q)) ++q;
    const char* e = eol;
    while (e > q && is_space(e[-1])) --e;
    p = eol + 1;
    if (q == e || word(q, e, "solid") || word(q, e, "endsolid") || word(q, e, "outer") || word(q, e, "endloop")) continue;
    StlEvent ev{kEvBadLine, {0.f, 0.f, 0.f}};
    if (word(q, e, "facet")) {
      ev.kind = kEvFacet;
    } else if (word(q, e, "endfacet")) {
      ev.kind = kEvEndFacet;
    } else if (word(q, e, "vertex")) {
      const char* r = q + 6;
      ev.kind = kEvVertex;
      for (int c = 0; c < 3; ++c) {
        double d;
        if (!parse_double(r, e, &d) || (r < e && !is_space(*r))) {
          ev.kind = kEvBadNumber;
          break;
        }
        ev.xyz[c] = f64_to_f32(d);
      }
      if (ev.kind == kEvVertex) {
        while (r < e && is_space(*r)) ++r;
        if (r != e) ev.kind = kEvBadLine;
      }
    }
    out->push_back(ev);
    if (ev.kind >= kEvBadLine) return;  // the first error of the chunk ends it
  }
}

int load_stl(const std::string& buf, const char* path, int n_threads, mvlm_mesh* m) {
  const uint8_t* data = reinterpret_cast<const uint8_t*>(buf.data());
  uint32_t nf = 0;
  std::vector<float> c;
  if (stl_is_binary(data, buf.size(), &nf)) {
    c.resize(static_cast<size_t>(nf) * 9);
    for (size_t t = 0; t < nf; ++t)
      for (int j = 0; j < 9; ++j) c[9 * t + static_cast<size_t>(j)] = read_coord(data + 84 + 50 * t + 12 + 4 * j, kFloat, false);
  } else {
    const std::vector<std::vector<StlEvent>> chunks =
        parallel_chunks<std::vector<StlEvent>>(buf.data(), buf.data() + buf.size(), n_threads, stl_lines);
    bool in_facet = false;
    int nvf = 0;
    for (const std::vector<StlEvent>& ch : chunks)
      for (const StlEvent& ev : ch) {
        MVLM_REQUIRE(ev.kind != kEvBadNumber, "mvlm_mesh_load: malformed ASCII number in %s", path);
        MVLM_REQUIRE(ev.kind != kEvBadLine, "mvlm_mesh_load: %s is neither a binary STL (84 + 50 n bytes) nor a valid ASCII STL",
                     path);
        if (ev.kind == kEvFacet) {
          MVLM_REQUIRE(!in_facet, "mvlm_mesh_load: malformed ASCII STL in %s (facet inside a facet)", path);
          in_facet = true;
          nvf = 0;
        } else if (ev.kind == kEvVertex) {
          MVLM_REQUIRE(in_facet && nvf < 3, "mvlm_mesh_load: malformed ASCII STL in %s (vertex outside a facet of 3)", path);
          c.insert(c.end(), ev.xyz, ev.xyz + 3);
          ++nvf;
        } else {
          MVLM_REQUIRE(in_facet && nvf == 3, "mvlm_mesh_load: malformed ASCII STL in %s (facet without 3 vertices)", path);
          in_facet = false;
        }
      }
    MVLM_REQUIRE(!in_facet, "mvlm_mesh_load: malformed ASCII STL in %s (unterminated facet)", path);
  }
  weld(c, m);
  return MVLM_OK;
}

bool has_suffix(const char* path, const char* suf) {
  const size_t n = strlen(path), k = strlen(suf);
  if (n < k) return false;
  for (size_t i = 0; i < k; ++i)
    if (static_cast<char>(tolower(static_cast<unsigned char>(path[n - k + i]))) != suf[i]) return false;
  return true;
}

}  // namespace
}  // namespace mvlm

using namespace mvlm;

extern "C" {

int mvlm_mesh_load(const char* path, int n_threads, mvlm_mesh** out) {
  MVLM_REQUIRE(path && out, "mvlm_mesh_load: null pointer");
  *out = nullptr;
  const bool ply = has_suffix(path, ".ply"), stl = has_suffix(path, ".stl");
  MVLM_REQUIRE(ply || stl, "mvlm_mesh_load: %s is not a .ply or .stl file", path);
  std::string buf;
  int rc = read_file(path, "mvlm_mesh_load", &buf);
  if (rc != MVLM_OK) return rc;
  mvlm_mesh* m = new mvlm_mesh();
  rc = ply ? load_ply(buf, path, n_threads, m) : load_stl(buf, path, n_threads, m);
  if (rc != MVLM_OK) {
    delete m;
    return rc;
  }
  if (m->verts.empty() || m->tris.empty()) {
    delete m;
    MVLM_REQUIRE(false, "File %s does not contain any points.", path);
  }
  *out = m;
  return MVLM_OK;
}

int mvlm_mesh_counts(const mvlm_mesh* m, int* n_verts, int* n_tris, int* has_colors) {
  MVLM_REQUIRE(m && n_verts && n_tris && has_colors, "mvlm_mesh_counts: null pointer");
  *n_verts = static_cast<int>(m->verts.size() / 3);
  *n_tris = static_cast<int>(m->tris.size() / 3);
  *has_colors = m->has_colors ? 1 : 0;
  return MVLM_OK;
}

int mvlm_mesh_copy(const mvlm_mesh* m, float* verts, uint8_t* colors, int32_t* tris) {
  MVLM_REQUIRE(m && verts && tris, "mvlm_mesh_copy: null pointer");
  memcpy(verts, m->verts.data(), m->verts.size() * sizeof(float));
  if (colors && m->has_colors) memcpy(colors, m->colors.data(), m->colors.size());
  memcpy(tris, m->tris.data(), m->tris.size() * sizeof(int32_t));
  return MVLM_OK;
}

void mvlm_mesh_free(mvlm_mesh* m) { delete m; }

}  // extern "C"
