// Stacked-hourglass heat-map CNN plan: the whole network as a static list of fused launches.
#pragma once
#include <map>
#include <string>
#include <vector>

#include "conv_umma.cuh"
#include "stages.cuh"

namespace mvlm {

// one state_dict entry: fp32 device tensor + its element count (checked against the layer's shape)
struct SdEntry {
  const float* p = nullptr;
  long long numel = -1;  // -1: unknown (not checked)
};
typedef std::map<std::string, SdEntry> StateDict;

// What one op computes, for the layer-wise tests (mvlm_debug_hourglass_ops): the state_dict names it applies and the
// plan buffer (allocation index, the same in both passes of emit()) and channel slice of every tensor it touches.
enum { kOpIn, kOpRes1, kOpRes2, kOpResUp, kOpOutPre, kOpOutRaw, kOpOutPost, kOpOutAux1, kOpOutAux2, kOpKeys,
       kOpOperands };
enum { kTermMid, kTermPre, kTermPost, kTermAux, kTermScale, kOpTerms };  // BatchNorm affines (pool / bnrelu: scale)
struct OpRecord {
  std::string layer, bias;  // conv: weight prefix ("hg1.rb5.conv2", "conv2.resample.2", "conv11"), bias key or ""
  int phase_a = -1, phase_b = -1;  // conv11 up-sampling phase
  struct Term { std::string bn; int off = 0; } terms[kOpTerms];  // BN name ("" = none) + channel offset into it
  int h = 0, w = 0, cin = 0, in_cs = 0, kh = 0, kw = 0, y_off0 = 0, x_off0 = 0, cout_pad = 0, n_tile = 0,
      cout_real = 0, pool2 = 0, aux_mode = 0;
  struct Operand { int buf = -1, cs = 0, co = 0; long long ws_off = -1; } opnd[kOpOperands];  // ws_off: real pass
};

struct NetOp {
  enum Kind { CONV, POOL, BNRELU, STEM, MEMSET, PEAKS } kind;  // STEM = image -> hi/lo bf16 staging
  ConvParams conv;  // CONV
  // eltwise / memset
  const __nv_bfloat16* in0 = nullptr;
  __nv_bfloat16* out_raw = nullptr;
  __nv_bfloat16* out_act = nullptr;
  const float* scale = nullptr;
  const float* shift = nullptr;
  int h = 0, w = 0, c = 0;
  size_t bytes = 0;
  bool is_head = false;  // conv11 phase: out_f32 patched per forward call
  const char* tag = "";
  OpRecord rec;
};

class HourglassNet {
 public:
  HourglassNet() = default;
  ~HourglassNet();
  // dry == true: only computes the workspace size (no CUDA calls).
  int build(const StateDict* sd, int n_landmarks, int cin, int n_views, int h, int w,
            void* workspace, size_t workspace_bytes, bool dry);
  int forward(const unsigned char* img_u8, const float* img_f32, float* out_heatmaps, float* out_peaks,
              cudaStream_t stream);
  int run_op(NetOp& op, const unsigned char* img_u8, const float* img_f32, float* out_heatmaps, float* out_peaks,
             cudaStream_t stream);
  // Captures the launch sequence of forward() into a CUDA graph per distinct argument tuple and replays it
  // (the plan is static: 144 launches per call).  Falls back to plain launches if capture is unavailable.
  int forward_graph(const unsigned char* img_u8, const float* img_f32, float* out_heatmaps, float* out_peaks,
                    cudaStream_t stream);

  // 0 = "simple" (arg-max), 1 = "moment" (paulsenpredictor.py:129-156) for the peaks forward() / forward_graph() write
  int set_selection_method(int method);
  // The network up to the fused arg-max: writes the (n_views x n_landmarks) u64 keys (ordered value << 32 | ~index)
  // into `out_keys` and runs no peak kernel (view-split path: out_keys is this rank's slot of the all-gather buffer).
  // Replays a CUDA graph like forward_graph.
  int forward_keys(const unsigned char* img_u8, const float* img_f32, unsigned long long* out_keys, cudaStream_t stream);

  // Debug aid: runs the plan `reps` times with a CUDA event pair around every op; ms_out[n_ops()] = mean ms per op.
  // roles_out (optional, n_ops() x 8 doubles): mean per-CTA role stall cycles of every conv op (conv_umma.cu).
  // trace_out (optional, kConvTraceTiles x 8 int64): per-tile timeline of CTA 0 of conv op `trace_op`.
  int profile_ops(const unsigned char* img_u8, const float* img_f32, float* out_peaks, int reps, float* ms_out,
                  double* roles_out, int trace_op, long long* trace_out, cudaStream_t stream);
  // one-line description of op i ("conv rb.conv 128x128 256->128 k3 pre res1 raw", "pool 64x64x256", ...)
  std::string describe_op(int i) const;

  // bytes and workspace offset of plan buffer i (allocation order)
  int n_buffers() const { return static_cast<int>(bufs_.size()); }
  size_t buffer_bytes(int i) const { return bufs_[i].bytes; }
  size_t buffer_offset(int i) const { return bufs_[i].offset; }

  size_t workspace_needed() const { return ws_needed_; }
  int n_views() const { return V_; }
  int n_landmarks() const { return L_; }
  int height() const { return H_; }
  int width() const { return W_; }
  double flops_per_view() const { return flops_; }
  int n_ops() const { return static_cast<int>(ops_.size()); }
  const std::vector<NetOp>& ops() const { return ops_; }
  std::vector<NetOp>& ops_mut() { return ops_; }
  // intermediate tensors exposed for layer-wise parity tests: name -> (ptr, h, w, c)
  struct Probe { const __nv_bfloat16* p; int h, w, c; };
  std::map<std::string, Probe> probes;

 private:
  struct T { __nv_bfloat16* p = nullptr; int h = 0, w = 0, c = 0; };
  T alloc(int h, int w, int c);
  void* ws_alloc(size_t bytes);
  // workspace packing, see ws_alloc in hourglass.cu
  struct Buf {
    size_t bytes = 0, fake_off = 0, offset = 0;
    int first = -1, last = -1;  // first / last op touching the buffer
    bool pinned = false;
  };
  int emit();
  void note_use(const void* p);
  void note_conv(const void* in, const ConvEpilogue& e);
  void assign_offsets();
  void probe(const char* name, const T& t);
  int param(const std::string& name, long long numel, size_t bytes, void** dst, const float** src);
  unsigned char* params_ = nullptr;  // one arena for packed weights / folded BatchNorm affines / biases
  size_t param_off_ = 0, param_cap_ = 0;
  cudaStream_t build_stream_ = nullptr;  // plan-build kernels (weight repacking) run here, not on the NULL stream
  static constexpr size_t kMaxGraphs = 8;
  std::vector<Buf> bufs_;
  size_t fake_off_ = 0, ws_needed_ = 0, next_buf_ = 0;
  bool layout_pass_ = false, keep_probes_ = false, reuse_ = true, fuse_elt_ = false;
  // parameter tensors (see param): null in the layout pass, filled on build_stream_ in the real pass
  int bn(const std::string& name, int c, const float** scale, const float** shift);
  int packed(const std::string& name, int cout, int cin, int k, int cout_pad, int cin_pad, const __nv_bfloat16** out);
  int bias(const std::string& name, int cout, int cout_pad, const float** out);
  int stem_weight(const __nv_bfloat16** out);
  int phase_weight(int a, int b, const __nv_bfloat16** out);
  // one convolution op: the first `cin` channels of `in` through the packed weights `w` (kh x kw taps, tap (0,0) at
  // input offset (y_off0, x_off0)); `flops` = the algorithmic FLOPs of the reference layer's share this op computes
  // `rec` carries the op's state_dict names; emit_conv adds the shape and the operands
  int emit_conv(const char* tag, T in, int cin, const __nv_bfloat16* w, int cout_pad, int n_tile, int kh, int kw,
                int y_off0, int x_off0, const ConvEpilogue& e, double flops, OpRecord rec, bool is_head = false);
  // operand `slot` of `r` is the workspace tensor at `p` (channel stride cs, first channel co); see OpRecord
  void record(OpRecord& r, int slot, const void* p, int cs, int co) const;
  void push_op(NetOp& op);
  std::vector<OpRecord> layout_recs_;  // the layout pass's records: buffer indices of the real pass's operands
  // pool_raw != nullptr: the block output is only consumed through a 2x2 max-pool (conv2 block, :410-411):
  // the three convs write the pooled raw tensor and relu(post_bn(pooled)) directly; no full-resolution output
  // up_low != nullptr: the nearest-x2 up-sampled half-resolution tensor is added to the block output
  // (hourglass up path, :334-359)
  // aux: copies of the block output for a second consumer, written by the block's own epilogues (ConvEpilogue::aux_mode):
  // mode 1 = relu(bn(y)) at full resolution -> *out1; mode 2 = max-pool(y) -> *out1 and relu(bn(max-pool(y))) -> *out2
  struct RbAux { int mode; const char* bn; T* out1; T* out2; };
  int rb(const std::string& p, T x, T a_in, T ar, int cin, int cout, const char* post_bn, T* post_act, T* y_out,
         T* pool_raw = nullptr, const T* up_low = nullptr, const RbAux* aux = nullptr);
  int hourglass(const std::string& p, T x, T a_x, T* out, const T* in_pooled = nullptr, const T* in_pooled_act = nullptr);
  int emit_pool(T in, T out_raw, const char* bn_name, T out_act);

  const StateDict* sd_ = nullptr;
  // state_dict entry `name` with exactly `numel` elements (a checkpoint of another model must not be misread)
  int sd_get(const std::string& name, long long numel, const float** out) const;
  int V_ = 0, H_ = 0, W_ = 0, L_ = 0, Lp_ = 0, cin_ = 0;
  uint8_t* ws_ = nullptr;
  size_t ws_size_ = 0;
  std::vector<void*> owned_;
  std::map<std::string, std::pair<float*, float*>> bn_cache_;  // folded BatchNorm scale / shift by name, per pass
  std::vector<NetOp> ops_;
  unsigned long long* keys_ = nullptr;
  unsigned long long* out_keys_ = nullptr;  // set for the duration of forward_keys
  int peak_method_ = 0;
  const __nv_bfloat16* phase_w_[4] = {nullptr, nullptr, nullptr, nullptr};  // conv11 phase kernels, bias, input
  const float* b11_ = nullptr;
  const __nv_bfloat16* x10_ = nullptr;
  double flops_ = 0.0;
  struct GraphKey { const void* a; const void* b; const void* c; const void* d; };
  std::vector<std::pair<GraphKey, cudaGraphExec_t>> graphs_;
};

}  // namespace mvlm
