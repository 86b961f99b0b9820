// Stacked-hourglass heat-map CNN as a static plan of fused launches (see hourglass.cuh).
//
// Dataflow of the reference model (src/mvlm/prediction/paulsenpredictor.py):
//   MVLMModel.forward :404-432, HourGlassModule.forward :301-361, ResidualBlock.forward :267-273,
//   eval mode (BatchNorm running statistics folded to scale/shift, dropout = identity).
// Only outputs[-1] (the conv11 branch) is consumed by the predictor (:204-205), so conv8 and its
// up-sampling (:418-419) are never scheduled.
//
// Every stored activation is NHWC bf16.  A ResidualBlock is three conv launches (+1 for the 1x1
// resample) whose epilogues write (i) the raw output into its channel slice of the block output
// with the residual slice added (torch.cat + residual, :273), (ii) the next conv's
// BatchNorm+ReLU'd input, and (iii) the BatchNorm+ReLU'd input of the block's designated consumer.
// conv11 on the nearest-x2 up-sampled conv10 output (:428-429) is evaluated as four 2x2 "phase"
// convolutions at the low resolution (taps that read the same low-res pixel are pre-summed), with
// the per-(view, landmark) arg-max fused into the epilogue, so the (V,L,256,256) fp32 heat maps
// (1.9 GB at V=100) are only materialised on request.
#include "hourglass.cuh"

#include <math.h>
#include <stdlib.h>

#include <algorithm>

namespace mvlm {

namespace {

__global__ void fold_bn_kernel(const float* w, const float* b, const float* m, const float* v, float eps, int n,
                               float* scale, float* shift) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float s = w[i] / sqrtf(v[i] + eps);
  scale[i] = s;
  shift[i] = b[i] - m[i] * s;
}

// OIHW fp32 -> [cout_pad][kw][kh][cin_pad] bf16
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, int cout, int cin, int kh, int kw,
                                        int cout_pad, int cin_pad, __nv_bfloat16* __restrict__ out) {
  const long long total = 1ll * cout_pad * kw * kh * cin_pad;
  for (long long i = blockIdx.x * 1ll * blockDim.x + threadIdx.x; i < total;
       i += 1ll * gridDim.x * blockDim.x) {
    const int ci = static_cast<int>(i % cin_pad);
    long long r = i / cin_pad;
    const int ky = static_cast<int>(r % kh);
    r /= kh;
    const int kx = static_cast<int>(r % kw);
    const int co = static_cast<int>(r / kw);
    float v = 0.f;
    if (co < cout && ci < cin) v = w[((1ll * co * cin + ci) * kh + ky) * kw + kx];
    out[i] = __float2bfloat16_rn(v);
  }
}

// conv3x3(nearest_up2(x)) phase (a,b): 2x2 taps at low resolution, [cout_pad][kx(2)][ky(2)][cin_pad] bf16.
//   a=0: rows {-1: w[0], 0: w[1]+w[2]}   a=1: rows {0: w[0]+w[1], +1: w[2]}   (same for columns with b)
__global__ void pack_phase_weight_kernel(const float* __restrict__ w, int cout, int cin, int a, int b, int cout_pad,
                                         int cin_pad, __nv_bfloat16* __restrict__ out) {
  const long long total = 1ll * cout_pad * 4 * cin_pad;
  for (long long i = blockIdx.x * 1ll * blockDim.x + threadIdx.x; i < total; i += 1ll * gridDim.x * blockDim.x) {
    const int ci = static_cast<int>(i % cin_pad);
    long long r = i / cin_pad;
    const int ky = static_cast<int>(r % 2);
    r /= 2;
    const int kx = static_cast<int>(r % 2);
    const int co = static_cast<int>(r / 2);
    float v = 0.f;
    if (co < cout && ci < cin) {
      const float* q = w + (1ll * co * cin + ci) * 9;
      // source rows / cols of the 3x3 kernel folded into this low-res tap
      const int r0 = a == 0 ? (ky == 0 ? 0 : 1) : (ky == 0 ? 0 : 2);
      const int r1 = a == 0 ? (ky == 0 ? 0 : 2) : (ky == 0 ? 1 : 2);
      const int c0 = b == 0 ? (kx == 0 ? 0 : 1) : (kx == 0 ? 0 : 2);
      const int c1 = b == 0 ? (kx == 0 ? 0 : 2) : (kx == 0 ? 1 : 2);
      for (int rr = r0; rr <= r1; ++rr)
        for (int cc = c0; cc <= c1; ++cc) v += q[rr * 3 + cc];
    }
    out[i] = __float2bfloat16_rn(v);
  }
}

// conv1.weight fp32 (co,cin,3,3) -> [co_pad][kx][ky][16] bf16 with the weights in channels 0..cin-1 (applied to
// the hi halves of the image) and again in 4..4+cin-1 (lo halves), see stem.cu
__global__ void pack_stem_weight_kernel(const float* __restrict__ w, int cout, int cin, int cout_pad,
                                        __nv_bfloat16* __restrict__ out) {
  const int total = cout_pad * 9 * 16;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int ch = i % 16;
    int r = i / 16;
    const int ky = r % 3;
    r /= 3;
    const int kx = r % 3;
    const int co = r / 3;
    const int ci = ch < 4 ? ch : (ch < 8 ? ch - 4 : -1);
    float v = 0.f;
    if (co < cout && ci >= 0 && ci < cin) v = w[((co * cin + ci) * 3 + ky) * 3 + kx];
    out[i] = __float2bfloat16_rn(v);
  }
}

__global__ void pad_bias_kernel(const float* b, int n, int n_pad, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pad) out[i] = i < n ? b[i] : 0.f;
}

inline int pad_to(int x, int m) { return (x + m - 1) / m * m; }

}  // namespace

int pack_conv_weight(const float* w_oihw, int cout, int cin, int kh, int kw, int cout_pad, int cin_pad,
                     __nv_bfloat16* out, cudaStream_t stream) {
  const long long total = 1ll * cout_pad * kw * kh * cin_pad;
  const int block = 256;
  const int grid = static_cast<int>((total + block - 1) / block > 4096 ? 4096 : (total + block - 1) / block);
  pack_conv_weight_kernel<<<grid, block, 0, stream>>>(w_oihw, cout, cin, kh, kw, cout_pad, cin_pad, out);
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

HourglassNet::~HourglassNet() {
  for (auto& g : graphs_) cudaGraphExecDestroy(g.second);
  for (void* p : owned_) cudaFree(p);
}

// Workspace allocation with buffer reuse.  emit() runs twice through the same calls: the LAYOUT pass (no CUDA calls)
// hands out fake, never-reused addresses, records for every buffer the first and the last op that touches it, and
// sizes the parameter arena; assign_offsets() then packs the buffers so that two share memory only when their
// lifetimes are disjoint (launches are stream-ordered, and programmatic dependent launch only overlaps a kernel's
// prologue, which touches no activation); the real pass hands out the packed addresses in the same allocation order,
// fills the parameters and plans the convolutions.  20.3 GB -> a few GB at 100 views of 256^2.
static uint8_t* const kFakeBase = reinterpret_cast<uint8_t*>(static_cast<uintptr_t>(1) << 44);

void* HourglassNet::ws_alloc(size_t bytes) {
  const size_t aligned = (bytes + 1023) & ~static_cast<size_t>(1023);
  if (layout_pass_) {
    Buf b;
    b.bytes = aligned;
    b.fake_off = fake_off_;
    bufs_.push_back(b);
    fake_off_ += aligned;
    return kFakeBase + b.fake_off;
  }
  if (ws_ == nullptr || next_buf_ >= bufs_.size()) return nullptr;
  return ws_ + bufs_[next_buf_++].offset;
}

// the op about to be pushed reads or writes the buffer `p` points into
void HourglassNet::note_use(const void* p) {
  if (!layout_pass_ || p == nullptr) return;
  const uint8_t* q = static_cast<const uint8_t*>(p);
  if (q < kFakeBase || q >= kFakeBase + fake_off_) return;
  const size_t off = static_cast<size_t>(q - kFakeBase);
  // buffers are in address order: last one starting at or before `off`
  size_t lo = 0, hi = bufs_.size();
  while (hi - lo > 1) {
    const size_t mid = (lo + hi) / 2;
    if (bufs_[mid].fake_off <= off) lo = mid; else hi = mid;
  }
  Buf& b = bufs_[lo];
  const int op = static_cast<int>(ops_.size());
  if (b.first < 0) b.first = op;
  b.last = std::max(b.last, op);
}

void HourglassNet::note_conv(const void* in, const ConvEpilogue& e) {
  note_use(in); note_use(e.out_pre); note_use(e.res1); note_use(e.res2); note_use(e.res_up); note_use(e.out_raw);
  note_use(e.out_post); note_use(e.argmax_keys); note_use(e.out_aux1); note_use(e.out_aux2);
}

void HourglassNet::assign_offsets() {
  const int n_ops = static_cast<int>(ops_.size());
  for (Buf& b : bufs_) {
    if (b.first < 0) { b.first = 0; b.last = n_ops; }  // never referenced by an op: keep it for the whole plan
    if (b.pinned || !reuse_) { b.first = 0; b.last = n_ops; }
  }
  // first-fit over a sorted free list, buffers taken in order of their first use
  std::vector<size_t> order(bufs_.size());
  for (size_t i = 0; i < order.size(); ++i) order[i] = i;
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return bufs_[a].first < bufs_[b].first; });
  struct Block { size_t off, bytes; };
  std::vector<Block> free_list;
  std::vector<size_t> live;
  size_t top = 0;
  auto release = [&](size_t id) {
    Block nb = {bufs_[id].offset, bufs_[id].bytes};
    size_t k = 0;
    while (k < free_list.size() && free_list[k].off < nb.off) ++k;
    free_list.insert(free_list.begin() + k, nb);
    for (size_t j = 0; j + 1 < free_list.size();) {  // coalesce neighbours
      if (free_list[j].off + free_list[j].bytes == free_list[j + 1].off) {
        free_list[j].bytes += free_list[j + 1].bytes;
        free_list.erase(free_list.begin() + j + 1);
      } else {
        ++j;
      }
    }
    if (!free_list.empty() && free_list.back().off + free_list.back().bytes == top) {  // give the tail back
      top = free_list.back().off;
      free_list.pop_back();
    }
  };
  for (size_t id : order) {
    Buf& b = bufs_[id];
    for (size_t j = 0; j < live.size();) {
      if (bufs_[live[j]].last < b.first) {
        release(live[j]);
        live.erase(live.begin() + j);
      } else {
        ++j;
      }
    }
    size_t best = free_list.size();
    for (size_t j = 0; j < free_list.size(); ++j)
      if (free_list[j].bytes >= b.bytes && (best == free_list.size() || free_list[j].bytes < free_list[best].bytes)) best = j;
    if (best < free_list.size()) {
      b.offset = free_list[best].off;
      free_list[best].off += b.bytes;
      free_list[best].bytes -= b.bytes;
      if (free_list[best].bytes == 0) free_list.erase(free_list.begin() + best);
    } else {
      b.offset = top;
      top += b.bytes;
    }
    ws_needed_ = std::max(ws_needed_, b.offset + b.bytes);
    ws_needed_ = std::max(ws_needed_, top);
    live.push_back(id);
  }
}

HourglassNet::T HourglassNet::alloc(int h, int w, int c) {
  T t;
  t.h = h; t.w = w; t.c = c;
  t.p = static_cast<__nv_bfloat16*>(ws_alloc(static_cast<size_t>(V_) * h * w * c * sizeof(__nv_bfloat16)));
  return t;
}

// Device memory for the plan's parameters (packed bf16 weights, folded BatchNorm affines, padded biases): sized in the
// layout pass, ONE cudaMalloc for the real pass (round 1 made 271 allocations and as many NULL-stream launches per plan).
// Every parameter tensor reserves its bytes here, by the same call in both passes, so the real pass's offsets are the
// ones the layout pass counted.  Layout pass: only the offset advances (*dst = *src = null).  Real pass: *dst = the
// tensor's slice of the arena, *src = state_dict entry `name` (`numel` elements), which the caller packs into *dst.
int HourglassNet::param(const std::string& name, long long numel, size_t bytes, void** dst, const float** src) {
  const size_t aligned = (bytes + 255) & ~static_cast<size_t>(255);
  *dst = (layout_pass_ || params_ == nullptr || param_off_ + aligned > param_cap_) ? nullptr : params_ + param_off_;
  *src = nullptr;
  param_off_ += aligned;
  if (layout_pass_) return MVLM_OK;
  const int rc = sd_get(name, numel, src);
  if (rc) return rc;
  MVLM_REQUIRE(*dst, "hourglass: parameter arena exhausted (%s)", name.c_str());
  return MVLM_OK;
}

int HourglassNet::sd_get(const std::string& name, long long numel, const float** out) const {
  auto f = sd_->find(name);
  MVLM_REQUIRE(f != sd_->end(), "hourglass: missing state_dict key %s", name.c_str());
  MVLM_REQUIRE(f->second.p != nullptr, "hourglass: null tensor for state_dict key %s", name.c_str());
  MVLM_REQUIRE(f->second.numel < 0 || f->second.numel == numel,
               "hourglass: size mismatch for %s: the checkpoint has %lld elements, this model (%d landmarks, %d image "
               "channels) needs %lld", name.c_str(), f->second.numel, L_, cin_, numel);
  *out = f->second.p;
  return MVLM_OK;
}

// a BatchNorm several convs apply is folded once per pass
int HourglassNet::bn(const std::string& name, int c, const float** scale, const float** shift) {
  auto it = bn_cache_.find(name);
  if (it == bn_cache_.end()) {
    void* buf;
    const float* src[4];
    int rc = param(name + ".weight", c, sizeof(float) * 2 * c, &buf, &src[0]);
    if (rc) return rc;
    float* f = static_cast<float*>(buf);
    if (!layout_pass_) {
      const char* suffix[3] = {".bias", ".running_mean", ".running_var"};
      for (int k = 0; k < 3; ++k)
        if ((rc = sd_get(name + suffix[k], c, &src[k + 1]))) return rc;
      fold_bn_kernel<<<ceil_div(c, 128), 128, 0, build_stream_>>>(src[0], src[1], src[2], src[3], 1e-5f, c, f, f + c);
      MVLM_CHECK_CUDA(cudaGetLastError());
    }
    it = bn_cache_.emplace(name, std::make_pair(f, f ? f + c : nullptr)).first;
  }
  *scale = it->second.first;
  *shift = it->second.second;
  return MVLM_OK;
}

int HourglassNet::packed(const std::string& name, int cout, int cin, int k, int cout_pad, int cin_pad,
                         const __nv_bfloat16** out) {
  void* buf;
  const float* src;
  const int rc = param(name, 1ll * cout * cin * k * k, sizeof(__nv_bfloat16) * cout_pad * k * k * cin_pad, &buf, &src);
  *out = static_cast<__nv_bfloat16*>(buf);
  if (rc || layout_pass_) return rc;
  return pack_conv_weight(src, cout, cin, k, k, cout_pad, cin_pad, static_cast<__nv_bfloat16*>(buf), build_stream_);
}

int HourglassNet::bias(const std::string& name, int cout, int cout_pad, const float** out) {
  void* buf;
  const float* src;
  const int rc = param(name, cout, sizeof(float) * cout_pad, &buf, &src);
  *out = static_cast<float*>(buf);
  if (rc || layout_pass_) return rc;
  pad_bias_kernel<<<ceil_div(cout_pad, 128), 128, 0, build_stream_>>>(src, cout, cout_pad, static_cast<float*>(buf));
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

// conv1.weight for the stem's 16-channel hi / lo input
int HourglassNet::stem_weight(const __nv_bfloat16** out) {
  void* buf;
  const float* src;
  const int rc = param("conv1.weight", 64ll * cin_ * 9, sizeof(__nv_bfloat16) * 64 * 9 * 16, &buf, &src);
  *out = static_cast<__nv_bfloat16*>(buf);
  if (rc || layout_pass_) return rc;
  pack_stem_weight_kernel<<<36, 256, 0, build_stream_>>>(src, 64, cin_, 64, static_cast<__nv_bfloat16*>(buf));
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

// conv11.weight folded into the 2x2 kernel of up-sampling phase (a, b)
int HourglassNet::phase_weight(int a, int b, const __nv_bfloat16** out) {
  void* buf;
  const float* src;
  const int rc = param("conv11.weight", 9ll * L_ * L_, sizeof(__nv_bfloat16) * Lp_ * 4 * Lp_, &buf, &src);
  *out = static_cast<__nv_bfloat16*>(buf);
  if (rc || layout_pass_) return rc;
  pack_phase_weight_kernel<<<64, 256, 0, build_stream_>>>(src, L_, L_, a, b, Lp_, Lp_, static_cast<__nv_bfloat16*>(buf));
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

int HourglassNet::emit_conv(const char* tag, T in, int cin, const __nv_bfloat16* w, int cout_pad, int n_tile, int kh,
                            int kw, int y_off0, int x_off0, const ConvEpilogue& e, double flops, bool is_head) {
  flops_ += flops;
  note_conv(in.p, e);
  NetOp op;
  op.kind = NetOp::CONV;
  op.tag = tag;
  op.is_head = is_head;
  op.h = in.h; op.w = in.w;
  if (!layout_pass_) {
    ConvShape s;
    s.in = in.p; s.n = V_; s.h = in.h; s.w = in.w; s.cin = cin; s.in_cs = in.c;
    s.wpacked = w; s.cout_pad = cout_pad; s.n_tile = n_tile; s.kh = kh; s.kw = kw;
    s.y_off0 = y_off0; s.x_off0 = x_off0;
    const int rc = conv_plan(s, e, &op.conv);
    if (rc) return rc;
  }
  ops_.push_back(op);
  return MVLM_OK;
}

int HourglassNet::rb(const std::string& p, T x, T a_in, T ar, int cin, int cout, const char* post_bn, T* post_act,
                     T* y_out, T* pool_raw, const T* up_low, const RbAux* aux) {
  const int h = a_in.h, w = a_in.w;
  T y = alloc(h, w, cout);
  T skip = x;
  int rc;
  if (cin != cout) {
    ConvEpilogue e;
    e.out_raw = y.p; e.raw_cs = cout; e.raw_co = 0;
    const __nv_bfloat16* wr;
    if ((rc = packed(p + ".resample.2.weight", cout, cin, 1, cout, cin, &wr)) ||
        (rc = emit_conv("rb.resample", ar, cin, wr, cout, cout < 128 ? cout : 128, 1, 1, 0, 0, e,
                        2.0 * cout * cin * ar.h * ar.w)))
      return rc;
    skip = y;  // the three convs accumulate in place
  }
  const float *ps = nullptr, *pt = nullptr;
  if (post_bn) {
    rc = bn(post_bn, cout, &ps, &pt);
    if (rc) return rc;
    *post_act = pool_raw ? alloc(h / 2, w / 2, cout) : alloc(h, w, cout);
  }
  if (pool_raw) *pool_raw = alloc(h / 2, w / 2, cout);
  // copies for a second consumer written by the three convs' epilogues (conv_umma.cuh, aux_mode)
  const float *as = nullptr, *at = nullptr;
  if (aux) {
    rc = bn(aux->bn, cout, &as, &at);
    if (rc) return rc;
    *aux->out1 = aux->mode == 2 ? alloc(h / 2, w / 2, cout) : alloc(h, w, cout);
    if (aux->mode == 2) *aux->out2 = alloc(h / 2, w / 2, cout);
  }
  const int c1 = cout / 2, c2 = cout / 4;
  // tightly packed intermediates (a 32-channel a2 in a 64-channel-stride buffer doubles its DRAM traffic); they die
  // with the block, and the packing reuses their memory
  T a1 = alloc(h, w, c1);
  T a2 = alloc(h, w, c2);
  const int widths[3] = {c1, c2, c2};
  const int offs[3] = {0, c1, c1 + c2};
  const int cins[3] = {cin, c1, c2};
  const T ins[3] = {a_in, a1, a2};
  const T pres[3] = {a1, a2, T()};
  const char* pre_bn[3] = {".bn2", ".bn3", nullptr};
  const char* names[3] = {".conv1", ".conv2", ".conv3"};
  for (int i = 0; i < 3; ++i) {
    ConvEpilogue e;
    if (pre_bn[i]) {
      rc = bn(p + pre_bn[i], widths[i], &e.pre_scale, &e.pre_shift);
      if (rc) return rc;
      e.out_pre = pres[i].p; e.pre_cs = pres[i].c; e.pre_co = 0;
    }
    e.res1 = skip.p; e.res1_cs = skip.c; e.res1_co = offs[i];
    if (up_low) { e.res_up = up_low->p; e.up_cs = up_low->c; e.up_co = offs[i]; }
    e.out_raw = pool_raw ? pool_raw->p : y.p; e.raw_cs = cout; e.raw_co = offs[i];
    e.pool2 = pool_raw != nullptr;
    if (post_bn) {
      e.post_scale = layout_pass_ ? nullptr : ps + offs[i];
      e.post_shift = layout_pass_ ? nullptr : pt + offs[i];
      e.out_post = post_act->p; e.post_cs = cout; e.post_co = offs[i];
    }
    if (aux) {
      e.aux_mode = aux->mode;
      e.aux_scale = layout_pass_ ? nullptr : as + offs[i];
      e.aux_shift = layout_pass_ ? nullptr : at + offs[i];
      e.out_aux1 = aux->out1->p; e.aux1_cs = cout; e.aux1_co = offs[i];
      if (aux->mode == 2) { e.out_aux2 = aux->out2->p; e.aux2_cs = cout; e.aux2_co = offs[i]; }
    }
    const int nt = widths[i] < 128 ? widths[i] : 128;
    const __nv_bfloat16* wc;
    if ((rc = packed(p + names[i] + ".weight", widths[i], cins[i], 3, widths[i], cins[i], &wc)) ||
        (rc = emit_conv("rb.conv", ins[i], cins[i], wc, widths[i], nt, 3, 3, -1, -1, e,
                        2.0 * widths[i] * cins[i] * 9 * h * w)))
      return rc;
  }
  *y_out = y;
  return MVLM_OK;
}

int HourglassNet::emit_pool(T in, T out_raw, const char* bn_name, T out_act) {
  note_use(in.p); note_use(out_raw.p); note_use(out_act.p);
  NetOp op;
  op.kind = NetOp::POOL;
  op.in0 = in.p; op.out_raw = out_raw.p; op.out_act = out_act.p;
  op.h = in.h; op.w = in.w; op.c = in.c;
  if (bn_name) {
    int rc = bn(bn_name, in.c, &op.scale, &op.shift);
    if (rc) return rc;
  }
  ops_.push_back(op);
  return MVLM_OK;
}

int HourglassNet::hourglass(const std::string& p, T x, T a_x, T* out, const T* in_pooled, const T* in_pooled_act) {
  // HourGlassModule.forward (:301-361).  The skip-branch blocks (rb1, rb3, rb5, rb7, rb9) are scheduled on the way
  // UP, after the low path of their level has returned, so that `F.interpolate(low, 2) + skip` (:334-359) is one
  // more residual of their epilogues instead of a separate elementwise pass over both tensors.  The max-pools on
  // the way DOWN (:309-329) are written by the epilogues of the block that produces their input (aux_mode 2): the
  // first one by the caller's block (in_pooled / in_pooled_act), the others by this level's down-path block.
  const int F = 256;
  int rc;
  T none;
  T lows[5], a_lows[5];
  T cur = x;
  const int low_blocks[5] = {2, 4, 6, 8, 10};
  const int skip_blocks[4] = {3, 5, 7, 9};
  T pooled, a;
  if (in_pooled) {
    pooled = *in_pooled;
    a = *in_pooled_act;
  }
  for (int lvl = 0; lvl < 5; ++lvl) {
    const std::string lb = p + ".rb" + std::to_string(low_blocks[lvl]);
    if (!(fuse_elt_ && (lvl > 0 || in_pooled))) {
      pooled = alloc(cur.h / 2, cur.w / 2, F);
      a = alloc(cur.h / 2, cur.w / 2, F);
      rc = emit_pool(cur, pooled, (lb + ".bn1").c_str(), a);
      if (rc) return rc;
    }
    const int nxt = lvl < 4 ? skip_blocks[lvl] : 11;
    const std::string post = p + ".rb" + std::to_string(nxt) + ".bn1";
    T next_pooled, next_a;
    const std::string next_bn = lvl < 4 ? p + ".rb" + std::to_string(low_blocks[lvl + 1]) + ".bn1" : "";
    RbAux aux = {2, next_bn.c_str(), &next_pooled, &next_a};
    rc = rb(lb, pooled, a, none, F, F, post.c_str(), &a_lows[lvl], &lows[lvl], nullptr, nullptr,
            (fuse_elt_ && lvl < 4) ? &aux : nullptr);
    if (rc) return rc;
    cur = lows[lvl];
    pooled = next_pooled;
    a = next_a;
  }
  T low2, a2, low3;
  rc = rb(p + ".rb11", cur, a_lows[4], none, F, F, (p + ".rb12.bn1").c_str(), &a2, &low2);
  if (rc) return rc;
  rc = rb(p + ".rb12", low2, a2, none, F, F, nullptr, nullptr, &low3);
  if (rc) return rc;
  cur = low3;
  const int ups[4][2] = {{13, 14}, {15, 16}, {17, 18}, {19, 20}};
  for (int lvl = 0; lvl < 4; ++lvl) {
    const std::string sb = p + ".rb" + std::to_string(skip_blocks[3 - lvl]);
    const std::string b1 = p + ".rb" + std::to_string(ups[lvl][0]);
    const std::string b2 = p + ".rb" + std::to_string(ups[lvl][1]);
    T s, a;
    rc = rb(sb, lows[3 - lvl], a_lows[3 - lvl], none, F, F, (b1 + ".bn1").c_str(), &a, &s, nullptr, &cur);
    if (rc) return rc;
    T l1, a1, l2;
    rc = rb(b1, s, a, none, F, F, (b2 + ".bn1").c_str(), &a1, &l1);
    if (rc) return rc;
    rc = rb(b2, l1, a1, none, F, F, nullptr, nullptr, &l2);
    if (rc) return rc;
    cur = l2;
  }
  T add5;
  rc = rb(p + ".rb1", x, a_x, none, F, F, nullptr, nullptr, &add5, nullptr, &cur);
  if (rc) return rc;
  *out = add5;
  return MVLM_OK;
}

int HourglassNet::build(const StateDict* sd, int n_landmarks, int cin, int n_views, int h,
                        int w, void* workspace, size_t workspace_bytes, bool dry) {
  MVLM_REQUIRE(n_landmarks > 0 && n_landmarks <= 128, "hourglass: n_landmarks=%d unsupported", n_landmarks);
  MVLM_REQUIRE(cin >= 1 && cin <= 4, "hourglass: image channels=%d unsupported", cin);
  MVLM_REQUIRE(n_views > 0 && h >= 64 && w >= 64 && h % 64 == 0 && w % 64 == 0,
               "hourglass: image size %dx%d must be a positive multiple of 64", h, w);
  MVLM_REQUIRE(dry || (sd && workspace), "hourglass: null state_dict/workspace");
  sd_ = sd;
  V_ = n_views; H_ = h; W_ = w; L_ = n_landmarks; cin_ = cin;
  Lp_ = pad_to(L_, 16);
  if (Lp_ == 112) Lp_ = 128;
  if (Lp_ == 48) Lp_ = 64;
  if (Lp_ == 16) Lp_ = 32;
  ws_ = static_cast<uint8_t*>(workspace); ws_size_ = workspace_bytes;
  // MVLM_HG_KEEP_PROBES=1: the probe tensors (layer-wise parity tests) keep their memory for the whole plan;
  // MVLM_HG_NO_REUSE=1: every buffer does (the round-1 layout, for A/B runs)
  keep_probes_ = getenv("MVLM_HG_KEEP_PROBES") != nullptr && atoi(getenv("MVLM_HG_KEEP_PROBES")) != 0;
  reuse_ = !(getenv("MVLM_HG_NO_REUSE") != nullptr && atoi(getenv("MVLM_HG_NO_REUSE")) != 0);
  // The hourglass max-pools and conv4's BatchNorm+ReLU copy are written by their producers' epilogues (aux_mode) instead
  // of stand-alone passes (155 -> 144 launches); MVLM_HG_ELT_FUSION=0 restores the passes.  History: in the first half of
  // round 2 the eleven passes it removes cost 0.58 ms (they run at 94 % of the HBM peak) and the producers, then
  // epilogue-bound, got 0.65 ms slower (profiles/r2_elt_fusion.txt); after the .ws / preamble / residual-prefetch work
  // the same switch measures 0.18 ms (1.1 %) faster, A/B on one box.
  fuse_elt_ = !(getenv("MVLM_HG_ELT_FUSION") != nullptr && atoi(getenv("MVLM_HG_ELT_FUSION")) == 0);
  // layout pass: lifetimes and packed offsets
  bufs_.clear(); fake_off_ = 0; ws_needed_ = 0; next_buf_ = 0;
  layout_pass_ = true;
  int rc = emit();
  layout_pass_ = false;
  if (rc) return rc;
  assign_offsets();
  if (dry) return MVLM_OK;
  MVLM_REQUIRE(ws_needed_ <= ws_size_, "hourglass: workspace too small (%zu needed, %zu given)", ws_needed_, ws_size_);
  // real pass: one arena for every parameter tensor, repacking kernels on a private stream (the state_dict tensors must
  // be complete when this is called: mvlm_b200/ops.py synchronises its stream before mvlm_hourglass_create)
  const size_t param_bytes = param_off_ + 4096;
  MVLM_CHECK_CUDA(cudaMalloc(&params_, param_bytes));
  owned_.push_back(params_);
  param_cap_ = param_bytes;
  MVLM_CHECK_CUDA(cudaStreamCreateWithFlags(&build_stream_, cudaStreamNonBlocking));
  rc = emit();
  if (rc == MVLM_OK && param_off_ > param_bytes) {
    set_error("hourglass: parameter arena overrun (%zu of %zu bytes)", param_off_, param_bytes);
    rc = MVLM_E_INVALID;
  }
  const cudaError_t ce = cudaStreamSynchronize(build_stream_);
  cudaStreamDestroy(build_stream_);
  build_stream_ = nullptr;
  if (rc) return rc;
  MVLM_CHECK_CUDA(ce);
  return MVLM_OK;
}

void HourglassNet::probe(const char* name, const T& t) {
  probes[name] = {t.p, t.h, t.w, t.c};
  if (layout_pass_ && keep_probes_ && t.p) {
    const size_t off = static_cast<size_t>(reinterpret_cast<const uint8_t*>(t.p) - kFakeBase);
    for (Buf& b : bufs_)
      if (b.fake_off == off) b.pinned = true;
  }
}

// emits the plan: ops_, probes, flops_, the parameter arena (layout pass: fake addresses, no CUDA calls)
int HourglassNet::emit() {
  const int h = H_, w = W_, cin = cin_;
  ops_.clear(); flops_ = 0.0; probes.clear();
  param_off_ = 0; bn_cache_.clear();
  int rc;
  const int F = 256, h2 = h / 2, w2 = w / 2;

  // ---- stem (:405-407): image -> hi/lo bf16 staging, then conv1 on the tensor cores with the fused
  //      bias -> bn1+ReLU -> {conv2.bn1, conv2.resample.0} BatchNorm+ReLU epilogue; conv2 block (:410)
  T a_c2 = alloc(h, w, 64), ar_c2 = alloc(h, w, 64);
  T img16 = alloc(h, w, 16);
  {
    note_use(img16.p);
    NetOp op;
    op.kind = NetOp::STEM;
    op.out_raw = img16.p; op.h = h; op.w = w; op.c = cin;
    ops_.push_back(op);
    const __nv_bfloat16* w1;
    ConvEpilogue e;
    if ((rc = stem_weight(&w1))) return rc;
    if ((rc = bias("conv1.bias", 64, 64, &e.bias))) return rc;
    if ((rc = bn("bn1", 64, &e.mid_scale, &e.mid_shift))) return rc;
    if ((rc = bn("conv2.bn1", 64, &e.pre_scale, &e.pre_shift))) return rc;
    if ((rc = bn("conv2.resample.0", 64, &e.post_scale, &e.post_shift))) return rc;
    e.out_pre = a_c2.p; e.pre_cs = 64; e.pre_co = 0;
    e.out_post = ar_c2.p; e.post_cs = 64; e.post_co = 0;
    if ((rc = emit_conv("conv1", img16, 16, w1, 64, 64, 3, 3, -1, -1, e, 2.0 * 64 * cin * 9 * h * w))) return rc;
  }
  T none, y2, y3, r3, a3, a4, a_h1, ar4;
  // conv2 block: its output is only consumed through the max-pool (:411) -> pooled outputs straight from the epilogues
  T x1;
  if ((rc = rb("conv2", none, a_c2, ar_c2, 64, 128, "conv3.bn1", &a3, &y2, &x1))) return rc;
  probe("x1", x1);
  if (fuse_elt_) {
    // conv4's resample branch reads relu(bn(y3)) (:263-265): a second act copy from the conv3 block's epilogues
    RbAux aux = {1, "conv4.resample.0", &ar4, nullptr};
    if ((rc = rb("conv3", x1, a3, none, 128, 128, "conv4.bn1", &a4, &y3, nullptr, nullptr, &aux))) return rc;
    probe("y3", y3);
  } else {
    if ((rc = rb("conv3", x1, a3, none, 128, 128, "conv4.bn1", &a4, &y3))) return rc;
    probe("y3", y3);
    ar4 = alloc(h2, w2, 128);
    note_use(y3.p); note_use(ar4.p);
    NetOp op;
    op.kind = NetOp::BNRELU;
    op.in0 = y3.p; op.out_act = ar4.p; op.h = h2; op.w = w2; op.c = 128;
    if ((rc = bn("conv4.resample.0", 128, &op.scale, &op.shift))) return rc;
    ops_.push_back(op);
  }
  // the first max-pool of each hourglass (:309) is written by the block that produces its input: conv4 / conv7
  T p1, pa1, p2, pa2;
  RbAux aux4 = {2, "hg1.rb2.bn1", &p1, &pa1};
  if ((rc = rb("conv4", y3, a4, ar4, 128, F, "hg1.rb1.bn1", &a_h1, &r3, nullptr, nullptr, fuse_elt_ ? &aux4 : nullptr))) return rc;
  probe("r3", r3);
  // ---- hourglass 1 (:414), conv5+bn2+relu (:416), conv6 (:417), conv7 + sum (:420-422)
  T hg1;
  if ((rc = hourglass("hg1", r3, a_h1, &hg1, fuse_elt_ ? &p1 : nullptr, fuse_elt_ ? &pa1 : nullptr))) return rc;
  probe("hg1", hg1);
  // conv5..conv10 read all channels of their input; their FLOPs count the true (unpadded) channels
  T ll1 = alloc(h2, w2, F);
  {
    ConvEpilogue e;
    const __nv_bfloat16* w5;
    if ((rc = bn("bn2", F, &e.pre_scale, &e.pre_shift))) return rc;
    e.out_pre = ll1.p; e.pre_cs = F; e.pre_co = 0;
    if ((rc = packed("conv5.weight", F, F, 3, F, F, &w5)) || (rc = bias("conv5.bias", F, F, &e.bias)) ||
        (rc = emit_conv("conv5", hg1, F, w5, F, 128, 3, 3, -1, -1, e, 2.0 * F * F * 9 * h2 * w2)))
      return rc;
  }
  T x6 = alloc(h2, w2, Lp_);
  {
    ConvEpilogue e;
    const __nv_bfloat16* w6;
    e.out_raw = x6.p; e.raw_cs = Lp_; e.raw_co = 0;
    if ((rc = packed("conv6.weight", L_, F, 3, Lp_, F, &w6)) || (rc = bias("conv6.bias", L_, Lp_, &e.bias)) ||
        (rc = emit_conv("conv6", ll1, F, w6, Lp_, Lp_, 3, 3, -1, -1, e, 2.0 * L_ * F * 9 * h2 * w2)))
      return rc;
  }
  T sum = alloc(h2, w2, F), a_h2;
  {
    ConvEpilogue e;
    e.res1 = r3.p; e.res1_cs = F; e.res1_co = 0;
    e.res2 = ll1.p; e.res2_cs = F; e.res2_co = 0;
    e.out_raw = sum.p; e.raw_cs = F; e.raw_co = 0;
    a_h2 = alloc(h2, w2, F);
    if ((rc = bn("hg2.rb1.bn1", F, &e.post_scale, &e.post_shift))) return rc;
    e.out_post = a_h2.p; e.post_cs = F; e.post_co = 0;
    if (fuse_elt_) {
      p2 = alloc(h2 / 2, w2 / 2, F);
      pa2 = alloc(h2 / 2, w2 / 2, F);
      if ((rc = bn("hg2.rb2.bn1", F, &e.aux_scale, &e.aux_shift))) return rc;
      e.aux_mode = 2;
      e.out_aux1 = p2.p; e.aux1_cs = F; e.aux1_co = 0;
      e.out_aux2 = pa2.p; e.aux2_cs = F; e.aux2_co = 0;
    }
    const __nv_bfloat16* w7;
    if ((rc = packed("conv7.weight", F, L_, 3, F, Lp_, &w7)) || (rc = bias("conv7.bias", F, F, &e.bias)) ||
        (rc = emit_conv("conv7", x6, Lp_, w7, F, 128, 3, 3, -1, -1, e, 2.0 * F * L_ * 9 * h2 * w2)))
      return rc;
  }
  probe("sum_temp", sum);
  // ---- hourglass 2 (:424), conv9+bn3+relu (:426), conv10 (:427)
  T hg2;
  if ((rc = hourglass("hg2", sum, a_h2, &hg2, fuse_elt_ ? &p2 : nullptr, fuse_elt_ ? &pa2 : nullptr))) return rc;
  T ll2 = alloc(h2, w2, F);
  {
    ConvEpilogue e;
    const __nv_bfloat16* w9;
    if ((rc = bn("bn3", F, &e.pre_scale, &e.pre_shift))) return rc;
    e.out_pre = ll2.p; e.pre_cs = F; e.pre_co = 0;
    if ((rc = packed("conv9.weight", F, F, 3, F, F, &w9)) || (rc = bias("conv9.bias", F, F, &e.bias)) ||
        (rc = emit_conv("conv9", hg2, F, w9, F, 128, 3, 3, -1, -1, e, 2.0 * F * F * 9 * h2 * w2)))
      return rc;
  }
  T x10 = alloc(h2, w2, Lp_);
  {
    ConvEpilogue e;
    const __nv_bfloat16* w10;
    e.out_raw = x10.p; e.raw_cs = Lp_; e.raw_co = 0;
    if ((rc = packed("conv10.weight", L_, F, 3, Lp_, F, &w10)) || (rc = bias("conv10.bias", L_, Lp_, &e.bias)) ||
        (rc = emit_conv("conv10", ll2, F, w10, Lp_, Lp_, 3, 3, -1, -1, e, 2.0 * L_ * F * 9 * h2 * w2)))
      return rc;
  }
  probe("x10", x10);
  // ---- conv11 on nearest-x2(conv10) (:428-429) as four 2x2 phase convs with fused arg-max
  keys_ = static_cast<unsigned long long*>(ws_alloc(sizeof(unsigned long long) * V_ * L_));
  {
    note_use(keys_);
    NetOp op;
    op.kind = NetOp::MEMSET;
    op.bytes = sizeof(unsigned long long) * V_ * L_;
    ops_.push_back(op);
  }
  if ((rc = bias("conv11.bias", L_, Lp_, &b11_))) return rc;
  x10_ = x10.p;
  for (int a = 0; a < 2; ++a) {
    for (int b = 0; b < 2; ++b) {
      ConvEpilogue e;
      e.bias = b11_;
      e.argmax_keys = keys_;
      e.cout_real = L_;
      e.up_sy = 2; e.up_sx = 2; e.up_py = a; e.up_px = b;
      // each phase computes a quarter of the reference conv11's output pixels
      if ((rc = phase_weight(a, b, &phase_w_[2 * a + b])) ||
          (rc = emit_conv("conv11.phase", x10, Lp_, phase_w_[2 * a + b], Lp_, Lp_, 2, 2, a - 1, b - 1, e,
                          2.0 * L_ * L_ * 9 * h2 * w2, true)))
        return rc;
    }
  }
  {
    note_use(keys_);
    note_use(x10.p);  // the "moment" selection re-evaluates windows of the last layer from its input
    NetOp op;
    op.kind = NetOp::PEAKS;
    ops_.push_back(op);
  }
  return MVLM_OK;
}

int HourglassNet::run_op(NetOp& op, const unsigned char* img_u8, const float* img_f32, float* out_heatmaps,
                         float* out_peaks, cudaStream_t stream) {
  // out_keys_ (forward_keys): the fused arg-max writes the caller's key buffer, e.g. this rank's slot of an
  // all-gather buffer, instead of the plan's own; no peak kernel runs here then
  unsigned long long* const keys = out_keys_ ? out_keys_ : keys_;
  switch (op.kind) {
    case NetOp::STEM:
      return image_to_hilo16(img_u8, img_f32, op.c, static_cast<size_t>(V_) * op.h * op.w, op.out_raw, stream);
    case NetOp::CONV:
      if (op.is_head) {
        ConvParams p = op.conv;
        p.e.out_f32 = out_heatmaps;
        p.e.argmax_keys = keys;
        return conv_launch(p, stream);
      }
      return conv_launch(op.conv, stream);
    case NetOp::POOL:
      return pool2_act(op.in0, V_, op.h, op.w, op.c, op.out_raw, op.scale, op.shift, op.out_act, stream);
    case NetOp::BNRELU:
      return bn_relu(op.in0, static_cast<size_t>(V_) * op.h * op.w, op.c, op.scale, op.shift, op.out_act, stream);
    case NetOp::MEMSET:
      MVLM_CHECK_CUDA(cudaMemsetAsync(keys, 0, op.bytes, stream));
      return MVLM_OK;
    case NetOp::PEAKS:
      if (out_peaks && !out_keys_) {
        if (peak_method_ == 1)
          return peaks_moment_from_keys(keys_, x10_, Lp_, Lp_, phase_w_, b11_, V_, L_, H_, W_, out_peaks, stream);
        return peaks_from_keys(keys_, V_, L_, H_, W_, out_peaks, stream);
      }
      return MVLM_OK;
  }
  return MVLM_OK;
}

int HourglassNet::set_selection_method(int method) {
  MVLM_REQUIRE(method == 0 || method == 1, "hourglass: unknown selection method %d", method);
  if (method != peak_method_) {
    for (auto& g : graphs_) cudaGraphExecDestroy(g.second);  // the captured launch sequences end in the other peak kernel
    graphs_.clear();
    peak_method_ = method;
  }
  return MVLM_OK;
}

int HourglassNet::forward_keys(const unsigned char* img_u8, const float* img_f32, unsigned long long* out_keys,
                               cudaStream_t stream) {
  MVLM_REQUIRE(out_keys, "hourglass: null key buffer");
  out_keys_ = out_keys;
  // graph key: the key buffer takes the place of the peak buffer (a distinct pointer tuple)
  const int rc = forward_graph(img_u8, img_f32, nullptr, reinterpret_cast<float*>(out_keys), stream);
  out_keys_ = nullptr;
  return rc;
}

int HourglassNet::forward(const unsigned char* img_u8, const float* img_f32, float* out_heatmaps, float* out_peaks,
                          cudaStream_t stream) {
  MVLM_REQUIRE(params_, "hourglass: forward on a dry plan");
  MVLM_REQUIRE(out_peaks || out_heatmaps, "hourglass: no output requested");
  for (NetOp& op : ops_) {
    const int rc = run_op(op, img_u8, img_f32, out_heatmaps, out_peaks, stream);
    if (rc != MVLM_OK) return rc;
  }
  return MVLM_OK;
}

int HourglassNet::profile_ops(const unsigned char* img_u8, const float* img_f32, float* out_peaks, int reps,
                              float* ms_out, double* roles_out, int trace_op, long long* trace_out,
                              cudaStream_t stream) {
  MVLM_REQUIRE(params_ && out_peaks && ms_out && reps > 0, "hourglass: bad profile_ops arguments");
  const size_t n = ops_.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) MVLM_CHECK_CUDA(cudaEventCreate(&e));
  for (size_t i = 0; i < n; ++i) ms_out[i] = 0.f;
  int rc = forward(img_u8, img_f32, nullptr, out_peaks, stream);  // warm-up
  for (int r = 0; r < reps && rc == MVLM_OK; ++r) {
    MVLM_CHECK_CUDA(cudaEventRecord(ev[0], stream));
    for (size_t i = 0; i < n && rc == MVLM_OK; ++i) {
      rc = run_op(ops_[i], img_u8, img_f32, nullptr, out_peaks, stream);
      MVLM_CHECK_CUDA(cudaEventRecord(ev[i + 1], stream));
    }
    MVLM_CHECK_CUDA(cudaStreamSynchronize(stream));
    for (size_t i = 0; i < n; ++i) {
      float ms = 0.f;
      MVLM_CHECK_CUDA(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
      ms_out[i] += ms / reps;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  if (roles_out && rc == MVLM_OK) {
    // one more pass with the conv kernel's role counters on: mean over the CTAs that ran (see conv_umma.cu)
    long long* dev = nullptr;
    MVLM_CHECK_CUDA(cudaMalloc(&dev, sizeof(long long) * kConvProfInts));
    std::vector<long long> host(kConvProfInts);
    for (size_t i = 0; i < n && rc == MVLM_OK; ++i) {
      for (int k = 0; k < 8; ++k) roles_out[i * 8 + k] = 0.0;
      if (ops_[i].kind == NetOp::CONV) {
        MVLM_CHECK_CUDA(cudaMemsetAsync(dev, 0, sizeof(long long) * kConvProfInts, stream));
        conv_set_profile_buffer(dev);
      }
      rc = run_op(ops_[i], img_u8, img_f32, nullptr, out_peaks, stream);
      conv_set_profile_buffer(nullptr);
      if (ops_[i].kind == NetOp::CONV && rc == MVLM_OK) {
        MVLM_CHECK_CUDA(cudaStreamSynchronize(stream));
        MVLM_CHECK_CUDA(cudaMemcpy(host.data(), dev, sizeof(long long) * kConvProfInts, cudaMemcpyDeviceToHost));
        if (trace_out && static_cast<int>(i) == trace_op)
          for (int k = 0; k < kConvTraceTiles * 16; ++k) trace_out[k] = host[kNumSMs * 8 + k];
        int ctas = 0;
        for (int c = 0; c < kNumSMs; ++c) {
          if (host[c * 8 + 4] == 0) continue;
          ++ctas;
          for (int k = 0; k < 8; ++k) roles_out[i * 8 + k] += static_cast<double>(host[c * 8 + k]);
        }
        for (int k = 0; k < 8; ++k) roles_out[i * 8 + k] /= ctas > 0 ? ctas : 1;
      }
    }
    cudaFree(dev);
  }
  return rc;
}

std::string HourglassNet::describe_op(int i) const {
  if (i < 0 || i >= static_cast<int>(ops_.size())) return "";
  const NetOp& op = ops_[i];
  char buf[256];
  switch (op.kind) {
    case NetOp::CONV: {
      const ConvShape& s = op.conv.s;
      const ConvEpilogue& e = op.conv.e;
      snprintf(buf, sizeof(buf), "conv %s %dx%d %d->%d k%d%s%s%s%s%s%s%s%s", op.tag, s.h, s.w, s.cin, s.cout_pad, s.kh,
               e.out_pre ? " pre" : "", e.res1 ? " res1" : "", e.res2 ? " res2" : "", e.res_up ? " up" : "", e.out_raw ? " raw" : "",
               e.out_post ? " post" : "", e.pool2 ? " pool" : (e.aux_mode == 2 ? " +pooled" : (e.aux_mode == 1 ? " +act2" : "")),
               e.argmax_keys ? " argmax" : "");
      break;
    }
    case NetOp::POOL: snprintf(buf, sizeof(buf), "pool %dx%dx%d", op.h, op.w, op.c); break;
    case NetOp::BNRELU: snprintf(buf, sizeof(buf), "bnrelu %dx%dx%d", op.h, op.w, op.c); break;
    case NetOp::STEM: snprintf(buf, sizeof(buf), "stem-stage %dx%dx%d", op.h, op.w, op.c); break;
    case NetOp::MEMSET: snprintf(buf, sizeof(buf), "memset %zu", op.bytes); break;
    case NetOp::PEAKS: snprintf(buf, sizeof(buf), "peaks"); break;
  }
  return buf;
}

int HourglassNet::forward_graph(const unsigned char* img_u8, const float* img_f32, float* out_heatmaps,
                                float* out_peaks, cudaStream_t stream) {
  for (auto& g : graphs_) {
    if (g.first.a == img_u8 && g.first.b == img_f32 && g.first.c == out_heatmaps && g.first.d == out_peaks) {
      MVLM_CHECK_CUDA(cudaGraphLaunch(g.second, stream));
      count_launch(static_cast<int>(ops_.size()));
      return MVLM_OK;
    }
  }
  // first call with these buffers: warm every kernel attribute outside capture, then capture
  int rc = forward(img_u8, img_f32, out_heatmaps, out_peaks, stream);
  if (rc != MVLM_OK) return rc;
  if (graphs_.size() >= kMaxGraphs) {  // many distinct buffer sets: the oldest graph makes room (never a silent fallback)
    cudaGraphExecDestroy(graphs_.front().second);
    graphs_.erase(graphs_.begin());
  }
  cudaGraph_t graph = nullptr;
  if (cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    return MVLM_OK;
  }
  rc = forward(img_u8, img_f32, out_heatmaps, out_peaks, stream);
  const cudaError_t ce = cudaStreamEndCapture(stream, &graph);
  if (rc != MVLM_OK || ce != cudaSuccess || !graph) {
    cudaGetLastError();
    if (graph) cudaGraphDestroy(graph);
    return rc;
  }
  cudaGraphExec_t exec = nullptr;
  if (cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess && exec) {
    graphs_.push_back({GraphKey{img_u8, img_f32, out_heatmaps, out_peaks}, exec});
    // the captured pass did not execute: run it once through the graph so that this call has its result
    MVLM_CHECK_CUDA(cudaGraphLaunch(exec, stream));
  } else {
    cudaGetLastError();
    rc = forward(img_u8, img_f32, out_heatmaps, out_peaks, stream);
  }
  cudaGraphDestroy(graph);
  return rc;
}

}  // namespace mvlm
