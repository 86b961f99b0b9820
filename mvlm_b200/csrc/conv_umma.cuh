// Implicit-GEMM convolution on tcgen05/TMEM fed by TMA (sm_100a).
//
// Replaces the torch.nn.Conv2d (+ BatchNorm2d + ReLU + residual add + cat)
// call sites of the reference CNN: paulsenpredictor.py:251-273 (ResidualBlock),
// :385-402 / :404-432 (MVLMModel top-level convs).
//
// Layout contract
//   activations : NHWC bf16, channel stride `cs` (elements) a multiple of 8;
//                 a conv reads `cin` channels (multiple of 16) starting at the
//                 base pointer.
//   weights     : packed bf16 [cout_pad][KW][KH][cin]  (K-major rows; one row
//                 per output channel; rows >= cout_real are zero).
//   GEMM view   : M = output channels (128 per CTA tile), N = output pixels (8 px x 32
//                 rows per CTA tile), K = KW*KH*cin.
#pragma once
#include "common.cuh"

namespace mvlm {

struct ConvEpilogue {
  const float* bias = nullptr;  // [cout_pad] fp32, added first
  // optional: v = relu(v*mid_scale+mid_shift) right after the bias (the stem's bn1+ReLU, paulsenpredictor.py:406-407)
  const float* mid_scale = nullptr;
  const float* mid_shift = nullptr;
  // act_pre = relu(v*pre_scale+pre_shift), v = acc+bias (BEFORE the residuals)
  const float* pre_scale = nullptr;
  const float* pre_shift = nullptr;
  __nv_bfloat16* out_pre = nullptr;
  int pre_cs = 0, pre_co = 0;
  // v += res1 + res2
  const __nv_bfloat16* res1 = nullptr;
  int res1_cs = 0, res1_co = 0;
  const __nv_bfloat16* res2 = nullptr;
  int res2_cs = 0, res2_co = 0;
  // v += res_up[(y/2, x/2)]: a half-resolution tensor added with nearest x2 up-sampling
  // (F.interpolate(scale_factor=2, mode="nearest") + skip, paulsenpredictor.py:334-359)
  const __nv_bfloat16* res_up = nullptr;
  int up_cs = 0, up_co = 0;
  // raw output (after residuals)
  __nv_bfloat16* out_raw = nullptr;
  int raw_cs = 0, raw_co = 0;
  // act_post = relu(v*post_scale+post_shift) (AFTER the residuals)
  const float* post_scale = nullptr;
  const float* post_shift = nullptr;
  __nv_bfloat16* out_post = nullptr;
  int post_cs = 0, post_co = 0;
  // Copies for a second consumer, written next to raw / post (the plan's stand-alone BatchNorm+ReLU and max-pool
  // passes fused into the producer, paulsenpredictor.py:263-265 and :309-329):
  //   aux_mode 1: out_aux1 = relu(v*aux_scale+aux_shift) at full resolution (a second act_post)
  //   aux_mode 2: out_aux1 = 2x2 max-pool of the bf16-rounded raw values, out_aux2 = relu(aux_scale*pooled+aux_shift),
  //               both at half resolution (needs even H and W); raw / post stay at full resolution
  int aux_mode = 0;
  const float* aux_scale = nullptr;
  const float* aux_shift = nullptr;
  __nv_bfloat16* out_aux1 = nullptr;
  int aux1_cs = 0, aux1_co = 0;
  __nv_bfloat16* out_aux2 = nullptr;
  int aux2_cs = 0, aux2_co = 0;
  // pool2: out_raw / out_post are written at HALF resolution: the 2x2 max-pool (F.max_pool2d(x, 2),
  // paulsenpredictor.py:411) of the bf16-rounded raw values, and relu(post_bn(pooled)); needs even H and W
  bool pool2 = false;
  // fp32 NCHW output (N, cout_real, H*up_sy, W*up_sx) at pixel (y*sy+py, x*sx+px)
  float* out_f32 = nullptr;
  // fused per-(image, channel) arg-max keys, see peaks.cu (atomicMax on u64)
  unsigned long long* argmax_keys = nullptr;
  int cout_real = 0;
  int up_sy = 1, up_sx = 1, up_py = 0, up_px = 0;
};

struct ConvShape {
  const __nv_bfloat16* in = nullptr;  // NHWC
  int n = 0, h = 0, w = 0;
  int cin = 0;    // channels read (multiple of 16)
  int in_cs = 0;  // channel stride of the input buffer
  const __nv_bfloat16* wpacked = nullptr;
  int cout_pad = 0;  // rows of wpacked; multiple of n_tile
  int n_tile = 0;    // 32, 64, 80, 96 or 128
  int kh = 3, kw = 3;
  int y_off0 = -1, x_off0 = -1;  // input offset of tap (0,0)
};

struct alignas(64) ConvParams {
  CUtensorMap tm_a;   // activations, 64-channel chunks (SWIZZLE_128B)
  CUtensorMap tm_b;   // weights,     64-channel chunks (SWIZZLE_128B)
  CUtensorMap tm_a2;  // tail chunk of `tail` (16 | 32) channels: SWIZZLE_32B | SWIZZLE_64B boxes
  CUtensorMap tm_b2;
  // residual inputs (res1, res2, res_up) as (channel slice, W, H, N) tensors: L2 prefetch boxes of one output tile
  CUtensorMap tm_r1, tm_r2, tm_up;
  int tail;           // cin % 64 if it is 16 or 32, else 0 (a 48-wide tail uses a zero-filled 64-wide box)
  ConvShape s;
  ConvEpilogue e;
  int tiles_x, tiles_y, n_nt, total_tiles;
  int tile_h;                             // rows of the 8-px-wide output tile: 32 (N = 256), 16, 8 or 4 for low maps
  int h_slot_bytes, n_hslots, n_wslots;   // operand ring geometry (conv_plan)
  int w_stationary;                       // 1: n_wslots = all weight tiles of the layer, loaded once per CTA
  // optional per-CTA cycle counters (8 x int64 per CTA), see conv_umma.cu "role timing"
  long long* prof;
  int debug_mode;  // 0 normal; 1 = MMA-only experiment (no TMA loads, operand waits skipped; results garbage)
};

// Builds the tensor maps and validates the shape.  Returns MVLM_* code.
int conv_plan(const ConvShape& s, const ConvEpilogue& e, ConvParams* out);
// Launches the persistent kernel for a planned conv.
int conv_launch(const ConvParams& p, cudaStream_t stream);
// OIHW fp32 weights -> the packed layout above, [cout_pad][kw][kh][cin_pad] bf16 with zero rows / channels past
// cout / cin (hourglass.cu).  Counts no launch: the plan build's packing is not part of a forward pass.
int pack_conv_weight(const float* w_oihw, int cout, int cin, int kh, int kw, int cout_pad, int cin_pad,
                     __nv_bfloat16* out, cudaStream_t stream);
// Debug: when non-null, the next conv_launch calls record role timings there (148 x 8 int64) followed by the
// per-tile timeline of CTA 0 (kConvTraceTiles x 16 int64, see conv_umma.cu).
constexpr int kConvTraceTiles = 64;
constexpr int kConvProfInts = 148 * 8 + kConvTraceTiles * 16;
void conv_set_profile_buffer(long long* dev_buf);
void conv_set_debug_mode(int mode);

}  // namespace mvlm
