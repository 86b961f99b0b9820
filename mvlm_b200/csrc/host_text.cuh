// Host-side text handling shared by the scan loaders obj_loader.cu and mesh_loader.cu: reading a whole file, the
// default thread count, the split of a text into line-aligned chunks parsed on one thread each, and the decimal rule.
#pragma once

#include <algorithm>
#include <charconv>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"

namespace mvlm {

// the whole file into *buf; `caller` prefixes the short-read message
inline int read_file(const char* path, const char* caller, std::string* buf) {
  FILE* fh = fopen(path, "rb");
  MVLM_REQUIRE(fh != nullptr, "File %s does not exist.", path);
  fseek(fh, 0, SEEK_END);
  const long size = ftell(fh);
  fseek(fh, 0, SEEK_SET);
  buf->assign(static_cast<size_t>(size > 0 ? size : 0), '\0');
  const size_t got = size > 0 ? fread(&(*buf)[0], 1, static_cast<size_t>(size), fh) : 0;
  fclose(fh);
  MVLM_REQUIRE(static_cast<long>(got) == size, "%s: short read on %s", caller, path);
  return MVLM_OK;
}

// n_threads <= 0: one per hardware thread, at most 16
inline int host_threads(int n_threads) {
  if (n_threads > 0) return n_threads;
  return static_cast<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
}

// chunk boundaries of [begin, end) at line starts, cuts[0] = begin and cuts[n] = end: one chunk below 64 KiB, else
// host_threads(n_threads), the i-th cut one past the first '\n' at or after max(begin + size * i / n, the previous cut)
inline std::vector<const char*> line_cuts(const char* begin, const char* end, int n_threads) {
  const size_t n = static_cast<size_t>(end - begin);
  n_threads = n < (1u << 16) ? 1 : host_threads(n_threads);
  std::vector<const char*> cuts(static_cast<size_t>(n_threads) + 1);
  cuts[0] = begin;
  for (int i = 1; i < n_threads; ++i) {
    const char* p = begin + n * static_cast<size_t>(i) / static_cast<size_t>(n_threads);
    if (p < cuts[static_cast<size_t>(i) - 1]) p = cuts[static_cast<size_t>(i) - 1];
    const char* nl = p < end ? static_cast<const char*>(memchr(p, '\n', static_cast<size_t>(end - p))) : nullptr;
    cuts[static_cast<size_t>(i)] = nl ? nl + 1 : end;
  }
  cuts[static_cast<size_t>(n_threads)] = end;
  return cuts;
}

// fn(chunk begin, chunk end, T* out) for every chunk of line_cuts, each on its own thread (chunk 0 on the caller's);
// the results in file order
template <class T, class F>
std::vector<T> parallel_chunks(const char* begin, const char* end, int n_threads, F&& fn) {
  const std::vector<const char*> cuts = line_cuts(begin, end, n_threads);
  const size_t k = cuts.size() - 1;
  std::vector<T> out(k);
  std::vector<std::thread> th;
  for (size_t i = 1; i < k; ++i) th.emplace_back([&, i] { fn(cuts[i], cuts[i + 1], &out[i]); });
  fn(cuts[0], cuts[1], &out[0]);
  for (auto& t : th) t.join();
  return out;
}

inline const char* skip_ws(const char* p, const char* end) {
  while (p < end && (*p == ' ' || *p == '\t' || *p == '\r')) ++p;
  return p;
}

// blanks, one optional '+' (from_chars rejects it, Python's float() accepts it), then std::from_chars: correctly
// rounded like Python's float()
inline bool parse_double(const char*& p, const char* end, double* out) {
  p = skip_ws(p, end);
  if (p < end && *p == '+') ++p;
  const auto r = std::from_chars(p, end, *out);
  if (r.ec != std::errc()) return false;
  p = r.ptr;
  return true;
}

}  // namespace mvlm
