// Native Wavefront OBJ scan loader (host code; SURVEY.md section 8(f) rank 1).
//
// Replaces vtkOBJReader as used by the reference's obj_to_actor (src/mvlm/utils/utils3d.py:16-21): positions
// `v x y z`, texture coordinates `vt u v`, faces `f a[/b[/c]] ...` (1-based or negative relative indices,
// polygons fan-triangulated).  Like vtkOBJReader, a position referenced with different `vt` indices is
// duplicated so that every output vertex has exactly one (position, uv) pair; output vertices are the
// unique (position index, uv index) pairs in ascending order, i.e. the same arrays, bit for bit, as the
// numpy restatement oracle/obj_ref.py::load_obj_python (the checker in tests/test_host_cpu.py).
//
// At ~50 scans/s on the GPU the text parse is the bottleneck of predict_one_file(path) (6 MB of text per
// scan; 1.05 s in numpy): the file is split at line boundaries into one chunk per thread, every chunk is
// parsed independently (std::from_chars: correctly rounded like Python's float(); both in host_text.cuh), and
// the chunks are concatenated in file order.
//
// With MVLM_OBJ_MATERIALS (mvlm_obj_load_ex) the loader also keeps the `mtllib` names, the distinct `usemtl` names in
// order of first appearance, and every triangle's material ordinal (the last `usemtl` before its `f` line; -1 before
// the first).  A chunk numbers only its own `usemtl` lines; the join offsets them by the lines of earlier chunks, and
// a chunk's triangles before its first `usemtl` inherit the last one of the chunks before it (DESIGN.md 7g).
#include <algorithm>
#include <charconv>
#include <cstdlib>
#include <cstring>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/mvlm_b200.h"
#include "common.cuh"
#include "host_text.cuh"

namespace mvlm {
namespace {

struct Chunk {
  std::vector<float> pos;     // xyz
  std::vector<float> tex;     // uv
  // face corners of this chunk, triangulated: (position index, uv index) as written in the file
  // (1-based / negative; resolved once the global counts are known), and the number of `v` / `vt`
  // lines seen in this chunk BEFORE each face (for negative indices)
  std::vector<long long> cv, ct;
  std::vector<int> v_before, vt_before;  // per triangle
  bool bad = false;
  // MVLM_OBJ_MATERIALS: this chunk's `usemtl` / `mtllib` names in file order, and per triangle the index of the last
  // `usemtl` line of this chunk before it (-1: none yet in this chunk)
  bool materials = false;
  std::vector<std::string> usemtl, mtllib;
  std::vector<int> mat_local;
};

// the rest of a `usemtl` / `mtllib` line, trimmed of blanks and a CR
inline std::string rest_trimmed(const char* p, const char* end) {
  p = skip_ws(p, end);
  while (end > p && (end[-1] == ' ' || end[-1] == '\t' || end[-1] == '\r')) --end;
  return std::string(p, static_cast<size_t>(end - p));
}

inline bool is_statement(const char* p, const char* eol, const char* word, size_t n) {
  return static_cast<size_t>(eol - p) > n && (p[n] == ' ' || p[n] == '\t') && memcmp(p, word, n) == 0;
}

inline bool parse_int(const char*& p, const char* end, long long* out) {
  auto r = std::from_chars(p, end, *out);
  if (r.ec != std::errc()) return false;
  p = r.ptr;
  return true;
}

void parse_chunk(const char* begin, const char* end, Chunk* c) {
  const char* p = begin;
  std::vector<long long> fv, ft;
  int n_v = 0, n_vt = 0;
  while (p < end) {
    const char* eol = static_cast<const char*>(memchr(p, '\n', static_cast<size_t>(end - p)));
    if (!eol) eol = end;
    if (eol - p >= 2 && p[0] == 'v' && p[1] == ' ') {
      const char* q = p + 2;
      double x, y, z;
      if (parse_double(q, eol, &x) && parse_double(q, eol, &y) && parse_double(q, eol, &z)) {
        c->pos.push_back(static_cast<float>(x));
        c->pos.push_back(static_cast<float>(y));
        c->pos.push_back(static_cast<float>(z));
        ++n_v;
      } else {
        c->bad = true;
      }
    } else if (eol - p >= 3 && p[0] == 'v' && p[1] == 't' && p[2] == ' ') {
      const char* q = p + 3;
      double u, v;
      if (parse_double(q, eol, &u) && parse_double(q, eol, &v)) {
        c->tex.push_back(static_cast<float>(u));
        c->tex.push_back(static_cast<float>(v));
        ++n_vt;
      } else {
        c->bad = true;
      }
    } else if (eol - p >= 2 && p[0] == 'f' && p[1] == ' ') {
      const char* q = p + 2;
      fv.clear();
      ft.clear();
      while (true) {
        q = skip_ws(q, eol);
        if (q >= eol) break;
        long long a = 0, b = 0;
        if (!parse_int(q, eol, &a)) { c->bad = true; break; }
        bool has_t = false;
        if (q < eol && *q == '/') {
          ++q;
          if (q < eol && *q != '/' && *q != ' ' && *q != '\t' && *q != '\r') {
            if (!parse_int(q, eol, &b)) { c->bad = true; break; }
            has_t = true;
          }
          if (q < eol && *q == '/') {  // normal index: ignored
            ++q;
            long long n;
            if (q < eol && *q != ' ' && *q != '\t' && *q != '\r') parse_int(q, eol, &n);
          }
        }
        fv.push_back(a);
        ft.push_back(has_t ? b : 0);  // 0 = no uv (OBJ indices are never 0)
      }
      for (size_t k = 1; k + 1 < fv.size(); ++k) {
        const size_t idx[3] = {0, k, k + 1};
        for (size_t j : idx) {
          c->cv.push_back(fv[j]);
          c->ct.push_back(ft[j]);
        }
        c->v_before.push_back(n_v);
        c->vt_before.push_back(n_vt);
        if (c->materials) c->mat_local.push_back(static_cast<int>(c->usemtl.size()) - 1);
      }
    } else if (c->materials && is_statement(p, eol, "usemtl", 6)) {
      c->usemtl.push_back(rest_trimmed(p + 7, eol));
    } else if (c->materials && is_statement(p, eol, "mtllib", 6)) {
      c->mtllib.push_back(rest_trimmed(p + 7, eol));
    }
    p = eol + 1;
  }
}

}  // namespace
}  // namespace mvlm

struct mvlm_obj {
  std::vector<float> verts, uvs;
  std::vector<int32_t> tris;
  bool has_uv = false;
  bool has_materials = false;                 // loaded with MVLM_OBJ_MATERIALS
  std::vector<int32_t> tri_material;          // per triangle: index into materials, -1 = none
  std::vector<std::string> materials, libraries;
};

using namespace mvlm;

extern "C" {

int mvlm_obj_load(const char* path, int n_threads, mvlm_obj** out) { return mvlm_obj_load_ex(path, n_threads, 0, out); }

int mvlm_obj_load_ex(const char* path, int n_threads, int flags, mvlm_obj** out) {
  MVLM_REQUIRE(path && out, "mvlm_obj_load: null pointer");
  MVLM_REQUIRE((flags & ~MVLM_OBJ_MATERIALS) == 0, "mvlm_obj_load_ex: unknown flags 0x%x", flags);
  const bool materials = (flags & MVLM_OBJ_MATERIALS) != 0;
  *out = nullptr;
  std::string buf;
  const int rc = read_file(path, "mvlm_obj_load", &buf);
  if (rc != MVLM_OK) return rc;
  const std::vector<Chunk> chunks = parallel_chunks<Chunk>(
      buf.data(), buf.data() + buf.size(), n_threads,
      [materials](const char* b, const char* e, Chunk* c) { c->materials = materials; parse_chunk(b, e, c); });
  size_t n_pos = 0, n_tex = 0, n_tri = 0;
  for (const Chunk& c : chunks) {
    MVLM_REQUIRE(!c.bad, "mvlm_obj_load: malformed v / vt / f line in %s", path);
    n_pos += c.pos.size() / 3;
    n_tex += c.tex.size() / 2;
    n_tri += c.v_before.size();
  }
  MVLM_REQUIRE(n_pos > 0, "File %s does not contain any points.", path);
  std::vector<float> pos(n_pos * 3), tex(n_tex * 2);
  // resolved 0-based corner indices: key = position << 32 | (uv + 1)   (uv + 1 == 0: no uv)
  std::vector<unsigned long long> keys(n_tri * 3);
  {
    size_t op = 0, ot = 0, ok = 0;
    bool any_uv = false;
    for (const Chunk& c : chunks) {
      for (size_t t = 0; t < c.v_before.size(); ++t) {
        // negative indices are relative to the elements read so far (OBJ specification)
        const long long v_seen = static_cast<long long>(op / 3) + c.v_before[t];
        const long long vt_seen = static_cast<long long>(ot / 2) + c.vt_before[t];
        for (int j = 0; j < 3; ++j) {
          const long long a = c.cv[t * 3 + static_cast<size_t>(j)], b = c.ct[t * 3 + static_cast<size_t>(j)];
          const long long vi = a > 0 ? a - 1 : v_seen + a;
          long long ti = -1;
          if (b != 0) ti = b > 0 ? b - 1 : vt_seen + b;
          MVLM_REQUIRE(vi >= 0 && vi < static_cast<long long>(n_pos), "mvlm_obj_load: face references vertex %lld of %zu in %s",
                       a, n_pos, path);
          MVLM_REQUIRE(ti >= -1 && ti < static_cast<long long>(n_tex), "mvlm_obj_load: face references vt %lld of %zu in %s", b, n_tex, path);
          if (ti >= 0) any_uv = true;
          keys[ok++] = (static_cast<unsigned long long>(vi) << 32) | static_cast<unsigned long long>(ti + 1);
        }
      }
      memcpy(pos.data() + op, c.pos.data(), c.pos.size() * sizeof(float));
      memcpy(tex.data() + ot, c.tex.data(), c.tex.size() * sizeof(float));
      op += c.pos.size();
      ot += c.tex.size();
    }
    mvlm_obj* o = new mvlm_obj();
    if (materials) {
      // usemtl line (file order) -> distinct name; triangles -> the last usemtl line before them
      o->has_materials = true;
      std::unordered_map<std::string, int32_t> ids;
      std::vector<int32_t> line_id;
      for (const Chunk& c : chunks) {
        for (const std::string& name : c.usemtl) {
          auto it = ids.emplace(name, static_cast<int32_t>(o->materials.size())).first;
          if (it->second == static_cast<int32_t>(o->materials.size())) o->materials.push_back(name);
          line_id.push_back(it->second);
        }
        o->libraries.insert(o->libraries.end(), c.mtllib.begin(), c.mtllib.end());
      }
      o->tri_material.reserve(n_tri);
      long long base = 0;  // usemtl lines of the chunks before this one
      for (const Chunk& c : chunks) {
        for (int local : c.mat_local) {
          const long long line = base + local;  // local = -1: the last line of the earlier chunks (or none)
          o->tri_material.push_back(line >= 0 ? line_id[static_cast<size_t>(line)] : -1);
        }
        base += static_cast<long long>(c.usemtl.size());
      }
    }
    o->tris.resize(n_tri * 3);
    if (n_tex == 0 || !any_uv) {
      // no texture coordinates in use: positions as they are, faces index them directly
      o->verts = std::move(pos);
      for (size_t i = 0; i < keys.size(); ++i) o->tris[i] = static_cast<int32_t>(keys[i] >> 32);
    } else {
      // unique (position, uv) pairs in ascending order without a comparison sort of all corners: counting sort by
      // position index, then each position's handful of uv indices is sorted / de-duplicated in place
      std::vector<uint32_t> start(n_pos + 1, 0);
      for (unsigned long long k : keys) ++start[static_cast<size_t>(k >> 32) + 1];
      for (size_t i = 0; i < n_pos; ++i) start[i + 1] += start[i];
      std::vector<uint32_t> bucket(keys.size());
      {
        std::vector<uint32_t> fill(start.begin(), start.end() - 1);
        for (unsigned long long k : keys) bucket[fill[static_cast<size_t>(k >> 32)]++] = static_cast<uint32_t>(k);
      }
      std::vector<uint32_t> ustart(n_pos + 1, 0);  // first output vertex of every position
      std::vector<uint32_t> ut;                     // uv index + 1 of every output vertex
      ut.reserve(n_pos + n_pos / 8);
      for (size_t v = 0; v < n_pos; ++v) {
        uint32_t* b0 = bucket.data() + start[v];
        uint32_t* b1 = bucket.data() + start[v + 1];
        std::sort(b0, b1);
        ustart[v] = static_cast<uint32_t>(ut.size());
        for (uint32_t* q = b0; q < b1; ++q)
          if (q == b0 || *q != q[-1]) ut.push_back(*q);
      }
      ustart[n_pos] = static_cast<uint32_t>(ut.size());
      const size_t n_out = ut.size();
      o->has_uv = true;
      o->verts.resize(n_out * 3);
      o->uvs.resize(n_out * 2);
      for (size_t v = 0; v < n_pos; ++v) {
        for (uint32_t i = ustart[v]; i < ustart[v + 1]; ++i) {
          memcpy(&o->verts[static_cast<size_t>(i) * 3], &pos[v * 3], 3 * sizeof(float));
          const long long ti = static_cast<long long>(ut[i]) - 1;
          o->uvs[static_cast<size_t>(i) * 2] = ti >= 0 ? tex[static_cast<size_t>(ti) * 2] : 0.f;
          o->uvs[static_cast<size_t>(i) * 2 + 1] = ti >= 0 ? tex[static_cast<size_t>(ti) * 2 + 1] : 0.f;
        }
      }
      for (size_t i = 0; i < keys.size(); ++i) {
        const size_t v = static_cast<size_t>(keys[i] >> 32);
        const uint32_t t1 = static_cast<uint32_t>(keys[i]);
        uint32_t j = ustart[v];
        while (ut[j] != t1) ++j;  // present by construction
        o->tris[i] = static_cast<int32_t>(j);
      }
    }
    *out = o;
  }
  return MVLM_OK;
}

int mvlm_obj_counts(const mvlm_obj* obj, int* n_verts, int* n_tris, int* has_uv) {
  MVLM_REQUIRE(obj && n_verts && n_tris && has_uv, "mvlm_obj_counts: null pointer");
  *n_verts = static_cast<int>(obj->verts.size() / 3);
  *n_tris = static_cast<int>(obj->tris.size() / 3);
  *has_uv = obj->has_uv ? 1 : 0;
  return MVLM_OK;
}

int mvlm_obj_copy(const mvlm_obj* obj, float* verts, float* uvs, int32_t* tris) {
  MVLM_REQUIRE(obj && verts && tris, "mvlm_obj_copy: null pointer");
  memcpy(verts, obj->verts.data(), obj->verts.size() * sizeof(float));
  if (uvs && obj->has_uv) memcpy(uvs, obj->uvs.data(), obj->uvs.size() * sizeof(float));
  memcpy(tris, obj->tris.data(), obj->tris.size() * sizeof(int32_t));
  return MVLM_OK;
}

int mvlm_obj_materials(const mvlm_obj* obj, int32_t* tri_material, int* n_materials, int* n_libraries) {
  MVLM_REQUIRE(obj && n_materials && n_libraries, "mvlm_obj_materials: null pointer");
  MVLM_REQUIRE(obj->has_materials, "mvlm_obj_materials: the scan was loaded without MVLM_OBJ_MATERIALS");
  *n_materials = static_cast<int>(obj->materials.size());
  *n_libraries = static_cast<int>(obj->libraries.size());
  if (tri_material) memcpy(tri_material, obj->tri_material.data(), obj->tri_material.size() * sizeof(int32_t));
  return MVLM_OK;
}

const char* mvlm_obj_material_name(const mvlm_obj* obj, int i) {
  if (!obj || i < 0 || static_cast<size_t>(i) >= obj->materials.size()) return nullptr;
  return obj->materials[static_cast<size_t>(i)].c_str();
}

const char* mvlm_obj_library_name(const mvlm_obj* obj, int i) {
  if (!obj || i < 0 || static_cast<size_t>(i) >= obj->libraries.size()) return nullptr;
  return obj->libraries[static_cast<size_t>(i)].c_str();
}

void mvlm_obj_free(mvlm_obj* obj) { delete obj; }

int mvlm_debug_obj_chunk_starts(const char* text, size_t len, int n_threads, long long* starts) {
  MVLM_REQUIRE((text || len == 0) && starts, "mvlm_debug_obj_chunk_starts: null pointer");
  const std::vector<const char*> cuts = line_cuts(text, text + len, n_threads);
  for (size_t i = 0; i + 1 < cuts.size(); ++i) starts[i] = cuts[i] - text;
  return static_cast<int>(cuts.size()) - 1;
}

}  // extern "C"
