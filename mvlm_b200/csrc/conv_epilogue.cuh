// Epilogue of the tcgen05 convolution kernel (conv_umma.cu): accumulator tile in TMEM -> bias / BatchNorm /
// ReLU / residuals / 2x2 max-pool / arg-max -> NHWC bf16 (or fp32 NCHW) stores.  See conv_umma.cu for the tile
// geometry and DESIGN.md section 4 for why it looks the way it does.
#pragma once
#include "conv_umma.cuh"

#include <type_traits>

namespace mvlm {
namespace epi {

constexpr int kThreads = 352;    // warps: 0 halo TMA, 1 MMA, 2..9 epilogue, 10 weight TMA
constexpr int kEpiWarps = 8;
constexpr int kTileW = 8;         // output tile: 8 px wide ...
constexpr int kMaxTileH = 32;     // ... and up to 32 rows high (N = 256)
constexpr int kMTile = 128;       // output channels per CTA tile (UMMA M)
constexpr int kStageFloats = 16 * 36;  // per-warp transpose buffer: 16 px x (32 ch + 4 pad)
constexpr int kMaxCout = 256;
constexpr int kTraceTiles = 64;   // debug timeline: tiles traced on CTA 0

// Epilogue feature flags (template parameter F): code for a feature is only generated when its bit is set,
// which keeps the per-row instruction count of the hot variants low (the epilogue is issue-bound).
enum : int { F_PRE = 1, F_RES1 = 2, F_RES2 = 4, F_RAW = 8, F_POST = 16, F_F32 = 32 /* fp32 NCHW map */, F_ARGMAX = 64,
              F_MID = 128 /* affine + ReLU right after the bias */, F_POOL = 256 /* raw/post at half resolution */,
              F_UP = 512 /* + nearest-x2 up-sampled half-resolution tensor */,
              F_M64 = 1024 /* cout <= 64: tcgen05.mma.ws with M = 64 / 32, the tile's pixels split over the TMEM lane groups */,
              F_POST2 = 2048 /* second full-resolution act copy (aux_mode 1) */,
              F_POOLX = 4096 /* additional pooled raw + pooled act copies (aux_mode 2) */,
              F_STAT = 8192 /* 3 x 3 taps over stationary weights: straight-line MMA issue */ };
constexpr int F_HEAD = F_F32 | F_ARGMAX;

// feature mask of a planned layer (without F_M64)
inline int feature_mask(const ConvEpilogue& e) {
  return (e.out_pre ? F_PRE : 0) | (e.res1 ? F_RES1 : 0) | (e.res2 ? F_RES2 : 0) | (e.out_raw ? F_RAW : 0) |
         (e.out_post ? F_POST : 0) | (e.out_f32 ? F_F32 : 0) | (e.argmax_keys ? F_ARGMAX : 0) |
         (e.mid_scale ? F_MID : 0) | (e.pool2 ? F_POOL : 0) | (e.res_up ? F_UP : 0) |
         (e.aux_mode == 1 ? F_POST2 : 0) | (e.aux_mode == 2 ? F_POOLX : 0);
}

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t order_f32(float f) {
  const uint32_t b = __float_as_uint(f);
  // negative: ~b, else b | 0x80000000  ==  b ^ (sign-extended sign | 0x80000000)
  return b ^ (static_cast<uint32_t>(static_cast<int32_t>(b) >> 31) | 0x80000000u);
}

__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]);
  __nv_bfloat162 b = __floats2bfloat162_rn(f[2], f[3]);
  __nv_bfloat162 c = __floats2bfloat162_rn(f[4], f[5]);
  __nv_bfloat162 d = __floats2bfloat162_rn(f[6], f[7]);
  uint4 r;
  r.x = *reinterpret_cast<uint32_t*>(&a);
  r.y = *reinterpret_cast<uint32_t*>(&b);
  r.z = *reinterpret_cast<uint32_t*>(&c);
  r.w = *reinterpret_cast<uint32_t*>(&d);
  return r;
}
// IEEE maximum that returns NaN when any input is NaN
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float fmax3_nan(float a, float b, float c) {
  float r;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// relu + round to bf16 in one instruction per pair (cvt.rn.relu.bf16x2.f32: first source -> upper half)
__device__ __forceinline__ uint32_t relu_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
// relu(f * s + t) -> bf16 x 8
__device__ __forceinline__ uint4 affine_relu_pack8(const float (&f)[8], const float (&sc)[8], const float (&sh)[8]) {
  uint4 r;
  r.x = relu_bf16x2(fmaf(f[0], sc[0], sh[0]), fmaf(f[1], sc[1], sh[1]));
  r.y = relu_bf16x2(fmaf(f[2], sc[2], sh[2]), fmaf(f[3], sc[3], sh[3]));
  r.z = relu_bf16x2(fmaf(f[4], sc[4], sh[4]), fmaf(f[5], sc[5], sh[5]));
  r.w = relu_bf16x2(fmaf(f[6], sc[6], sh[6]), fmaf(f[7], sc[7], sh[7]));
  return r;
}
__device__ __forceinline__ void add8(const uint4& q, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = __bfloat1622float2(h[j]);
    f[2 * j] += t.x;
    f[2 * j + 1] += t.y;
  }
}
__device__ __forceinline__ uint4 max_bf16x8(const uint4& a, const uint4& b) {
  uint4 r;
  const __nv_bfloat162* pa = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* pb = reinterpret_cast<const __nv_bfloat162*>(&b);
  __nv_bfloat162* pr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) pr[j] = __hmax2(pa[j], pb[j]);
  return r;
}
__device__ __forceinline__ void lds8(const float* src, float (&v)[8]) {
  const float4 a = reinterpret_cast<const float4*>(src)[0];
  const float4 b = reinterpret_cast<const float4*>(src)[1];
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}

// role timing: wait on an mbarrier and add the stalled cycles to `acc` when profiling is on.  The wait is the bounded one
// WITHOUT the printf: a call in the loop makes every value that is live across it caller-saved, and the MMA thread then
// re-materialises its descriptors in uniform registers (seven R2UR) on every tap
__device__ __forceinline__ void timed_wait(uint64_t* b, uint32_t parity, bool prof, long long& acc) {
  if (!prof) { ptx::mbar_wait_trap(b, parity); return; }
  const long long t0 = clock64();
  ptx::mbar_wait_trap(b, parity);
  acc += clock64() - t0;
}

struct TileCoord {
  int mt, tx, ty, img;
};

// Per-output-channel parameter arrays in shared memory, never null, at least cout_pad long.
struct ChannelParams {
  const float* bias;
  const float* mid_s;  // F_MID parameters, or the aux_scale / aux_shift of F_POST2 / F_POOLX (never both)
  const float* mid_t;
  const float* pre_s;
  const float* pre_t;
  const float* post_s;
  const float* post_t;
};

// running arg-max of the F_ARGMAX variants (lane = channel), flushed when the CTA moves to another image
struct ArgmaxState {
  uint32_t best_hi = 0u, best_lo = 0u;
  int cur_img = -1;
};

// optional per-tile timeline of one epilogue warp (see conv_umma.cu)
struct EpiTrace {
  long long* trace = nullptr;
  int trace_i = 0;
  long long t0 = 0;
  bool on = false;  // this thread records
};
#define MVLM_EPI_TRACE(slot)                                                                              \
  do {                                                                                                    \
    if (tr.on && tr.trace && tr.trace_i < kTraceTiles) tr.trace[tr.trace_i * 16 + (slot)] = clock64() - tr.t0; \
  } while (0)

// One accumulator tile.  Pixel n of the tile = 8 * (row in tile) + (pixel in row).  One "unit" (one TMEM load,
// one transpose) = 16 pixels = 2 image rows x 8 px of the warp's 32 channels.
//   M = 128 (plain tcgen05.mma): TMEM lane = output channel, TMEM column = pixel n.
//   F_M64 (tcgen05.mma.ws, cout <= 64): the tile is spread over all 128 lanes (ptx::umma_ws_bf16) --
//     M = 64: lane group g = channels 32 * (g % 2) .., pixels (g / 2) * N/2 + column,
//     M = 32: lane group g = channels 0 .. 31,         pixels g * N/4 + column
//     -- so every epilogue warp holds 32 channels in its 32 lanes, like at M = 128, and the lane groups that hold the
//     same channels ("replicas") split the tile's pixel rows.
// The epilogue is latency-bound (two warps per scheduler, dependent TMEM -> shared -> registers -> global chain
// per unit), so fewer, fatter units matter.
//
// `tmem_acc` = TMEM address of column 0 of this tile's accumulator stage; `t_full` / `parity` = the barrier the
// MMA warp commits to.  The caller releases the stage (tcgen05 fence + arrive on its t_empty barrier) afterwards.
template <int F>
__device__ __forceinline__ void epilogue_tile(const ConvShape& s, const ConvEpilogue& e, const int tile_h,
                                              const ChannelParams& ep, const TileCoord& tc,
                                              uint64_t* t_full, const uint32_t parity, const uint32_t tmem_acc,
                                              float* stage, const int ew, const int lane_grp, const int lane,
                                              ArgmaxState& am, const bool prof, long long& w0, EpiTrace& tr) {
  constexpr bool WS = (F & F_M64) != 0;
  constexpr int kM = kMTile;
  constexpr int kChGrp = 32;                 // channels per TMEM lane group
  constexpr int kPitch = 36;                 // floats per pixel row of the transpose buffer
  constexpr int kCols = 16;                  // accumulator columns per unit
  constexpr int kUnitRows = kCols / 8;       // image rows per unit
  static_assert(kCols * kPitch <= kStageFloats, "transpose buffer");
  // F_M64: `rep` = 2 (M = 64: 33 .. 64 channels) or 4 (M = 32) lane groups hold the same channels and different pixel
  // rows of the tile.  A shift count, so that the per-tile index arithmetic below needs no integer division.
  const int rep_log2 = !WS ? 0 : (s.cout_pad <= 32 ? 2 : 1);
  // ew = index of this epilogue warp (0..7), lane_grp = its hardware warp id % 4: the TMEM lanes it may read are
  // 32 * lane_grp ..
  const int n_cgrp = 4 >> rep_log2;  // distinct channel groups along M
  const int cgrp = lane_grp & (n_cgrp - 1);
  const int replica = lane_grp >> (2 - rep_log2);
  const int n_units = max(1, tile_h / kUnitRows);
  const int upr = max(1, n_units >> rep_log2);              // units per replica (= TMEM columns / 16 of the tile)
  const int upw = max(1, upr >> 1);                         // units per warp (two warps share a lane group)
  const int u_local = (ew >> 2) * upw;                      // my first unit among my replica's
  const int u_begin = replica * upr + u_local;              // ... and among the tile's
  const int oh = s.h * e.up_sy, ow = s.w * e.up_sx;
  // channel-major role (TMEM load, bias, transpose store): lane = channel.
  // pixel-major role after the transpose, two passes per unit:
  //   lane -> (pixel column pj = lane/4, channels (lane%4)*8 .. +7), unit row ip in pass ip
  const int pj = lane >> 2;
  const int cq = (lane & 3) * 8;
  constexpr bool kBf16Out = (F & (F_PRE | F_RAW | F_POST)) != 0;
  // byte strides of one image row in every tensor the epilogue touches: an access of unit r, pass ip is then
  // (per-tile base pointer) + (kUnitRows * r + ip) * stride with a compile-time row offset
  const uint32_t rs_pre = static_cast<uint32_t>(s.w * e.pre_cs) * 2u, rs_res1 = static_cast<uint32_t>(s.w * e.res1_cs) * 2u;
  const uint32_t rs_res2 = static_cast<uint32_t>(s.w * e.res2_cs) * 2u;
  const uint32_t rs_up = static_cast<uint32_t>((s.w >> 1) * e.up_cs) * 2u;
  // F_POOL: raw / post live at half resolution
  const uint32_t rs_raw = static_cast<uint32_t>(((F & F_POOL) ? (s.w >> 1) : s.w) * e.raw_cs) * 2u;
  const uint32_t rs_post = static_cast<uint32_t>(((F & F_POOL) ? (s.w >> 1) : s.w) * e.post_cs) * 2u;
  const uint32_t rs_aux1 = static_cast<uint32_t>(((F & F_POOLX) ? (s.w >> 1) : s.w) * e.aux1_cs) * 2u;
  const uint32_t rs_aux2 = static_cast<uint32_t>((s.w >> 1) * e.aux2_cs) * 2u;
  // Residual inputs do not depend on the accumulator: they are fetched in BATCHES before they are needed -- all
  // units of a tile while its MMAs still run when they fit in ~64 registers, else half of them then and the other
  // half once the first are consumed.  (Loads issued one by one while earlier ones are being consumed do not work:
  // the few hardware scoreboards are shared, so every use then waits for the newest load; measured.)
  constexpr bool kHasRes = (F & (F_RES1 | F_RES2 | F_UP)) != 0;
  constexpr int kMaxUpw = WS ? 4 : 8;  // units per warp at N = 256
  constexpr int kResRegs = 4 * (2 * (((F & F_RES1) ? 1 : 0) + ((F & F_RES2) ? 1 : 0)) + ((F & F_UP) ? 1 : 0));
  constexpr int kResBudget = 64;
  constexpr int kPref = !kHasRes ? 1 : (kResRegs * kMaxUpw <= kResBudget ? kMaxUpw : (kResRegs * kMaxUpw <= 2 * kResBudget ? kMaxUpw / 2 : (kMaxUpw >= 4 ? kMaxUpw / 4 : 1)));  // units per batch
  uint4 r1[kPref][2], r2[(F & F_RES2) ? kPref : 1][2], ru[(F & F_UP) ? kPref : 1][1];

  const int m0 = tc.mt * kM;
  const int c_lane = m0 + cgrp * kChGrp + lane;       // channel-major role: my output channel
  const int c0 = m0 + cgrp * kChGrp + cq;             // pixel-major role: first of my 8 channels
  const bool grp_active = m0 + cgrp * kChGrp < s.cout_pad;
  const int y_first = tc.ty * tile_h + kUnitRows * u_begin;  // first image row handled by this warp
  const bool rows_active = u_local < upr && y_first < s.h;
  const bool ch_ok = c0 < s.cout_pad;  // weight rows beyond cout_pad are never loaded
  const int xa = tc.tx * kTileW + pj;
  const bool vx = ch_ok && xa < s.w;
  // PIXEL index of my pixel in pass 0 of the first unit: (tc.img, y_first, xa); 32-bit (checked in conv_plan),
  // widened before it is multiplied with a channel stride
  auto pix = [&]() __attribute__((always_inline)) { return (static_cast<uint32_t>(tc.img) * s.h + y_first) * s.w + xa; };
  // element index of the half-resolution pixel (tc.img, y_first/2, xa/2): F_POOL outputs, F_UP input
  auto ppix = [&]() __attribute__((always_inline)) {
    return (static_cast<uint32_t>(tc.img) * (s.h >> 1) + (y_first >> 1)) * (s.w >> 1) + (xa >> 1);
  };
  if ((F & F_ARGMAX) && tc.img != am.cur_img) {
    if (am.cur_img >= 0 && am.best_hi != 0u && c_lane < e.cout_real)
      atomicMax(e.argmax_keys + static_cast<size_t>(am.cur_img) * e.cout_real + c_lane,
                (static_cast<unsigned long long>(am.best_hi) << 32) | am.best_lo);
    am.best_hi = 0u; am.best_lo = 0u;
    am.cur_img = tc.img;
  }
  // per-tile base pointers of my (pixel, 8 channels) in the first unit
  uint8_t* const b_pre = (F & F_PRE) ? reinterpret_cast<uint8_t*>(e.out_pre + e.pre_co + c0 + static_cast<size_t>(pix()) * e.pre_cs) : nullptr;
  uint8_t* const b_raw = (F & F_RAW) ? reinterpret_cast<uint8_t*>(e.out_raw + e.raw_co + c0 + static_cast<size_t>((F & F_POOL) ? ppix() : pix()) * e.raw_cs) : nullptr;
  uint8_t* const b_post = (F & F_POST) ? reinterpret_cast<uint8_t*>(e.out_post + e.post_co + c0 + static_cast<size_t>((F & F_POOL) ? ppix() : pix()) * e.post_cs) : nullptr;
  uint8_t* const b_aux1 = (F & (F_POST2 | F_POOLX)) ? reinterpret_cast<uint8_t*>(e.out_aux1 + e.aux1_co + c0 + static_cast<size_t>((F & F_POOLX) ? ppix() : pix()) * e.aux1_cs) : nullptr;
  uint8_t* const b_aux2 = (F & F_POOLX) ? reinterpret_cast<uint8_t*>(e.out_aux2 + e.aux2_co + c0 + static_cast<size_t>(ppix()) * e.aux2_cs) : nullptr;
  // rows at / below my first pixel that exist in the image (0 when my pixel column / channels do not):
  // unit r, pass ip is valid iff kUnitRows * r + ip < n_rows_ok
  const int n_rows_ok = vx ? s.h - y_first : 0;
  const uint8_t* const b_res1 = (F & F_RES1) ? reinterpret_cast<const uint8_t*>(e.res1 + e.res1_co + c0 + static_cast<size_t>(pix()) * e.res1_cs) : nullptr;
  const uint8_t* const b_res2 = (F & F_RES2) ? reinterpret_cast<const uint8_t*>(e.res2 + e.res2_co + c0 + static_cast<size_t>(pix()) * e.res2_cs) : nullptr;
  const uint8_t* const b_up = (F & F_UP) ? reinterpret_cast<const uint8_t*>(e.res_up + e.up_co + c0 + static_cast<size_t>(ppix()) * e.up_cs) : nullptr;
  auto prefetch_batch = [&](int u0) __attribute__((always_inline)) {  // units u0 .. u0 + kPref - 1 (u0 compile-time after unrolling)
#pragma unroll
    for (int q = 0; q < kPref; ++q) {
      const int u = u0 + q;
      if (u < upw) {
#pragma unroll
        for (int ip = 0; ip < 2; ++ip) {
          const int row = kUnitRows * u + ip;
          if (row < n_rows_ok) {
            if (F & F_RES1) r1[q][ip] = *reinterpret_cast<const uint4*>(b_res1 + static_cast<size_t>(row * rs_res1));
            if (F & F_RES2) r2[q][ip] = *reinterpret_cast<const uint4*>(b_res2 + static_cast<size_t>(row * rs_res2));
            // nearest x2: rows 2k, 2k+1 and columns xa, xa^1 all read low-res pixel (k, xa/2);
            // both passes share one low-res row per unit
            if ((F & F_UP) && ip == 0)
              ru[q][0] = *reinterpret_cast<const uint4*>(b_up + static_cast<size_t>((row >> 1) * rs_up));
          }
        }
      }
    }
  };
  if (kHasRes && grp_active && rows_active) prefetch_batch(0);
  // per-channel parameters of my 8 channels (pixel-major role) and my channel (channel-major role)
  float pre_s[8], pre_t[8], post_s[8], post_t[8];
  const int c0_ok = ch_ok ? c0 : 0;
  if (F & F_PRE) { lds8(ep.pre_s + c0_ok, pre_s); lds8(ep.pre_t + c0_ok, pre_t); }
  if (F & F_POST) { lds8(ep.post_s + c0_ok, post_s); lds8(ep.post_t + c0_ok, post_t); }
  const int c_lane_ok = c_lane < s.cout_pad ? c_lane : 0;
  const float bias_c = ep.bias[c_lane_ok];
  const float mid_s_c = ep.mid_s[c_lane_ok], mid_t_c = ep.mid_t[c_lane_ok];
  MVLM_EPI_TRACE(7);  // residual prefetch issued, parameters loaded, about to wait
  timed_wait(t_full, parity, prof, w0);
  ptx::tc_fence_after();
  MVLM_EPI_TRACE(5);
  if (grp_active && rows_active) {
    // TMEM column of my first unit: the tile's own pixel index at M = 128, the index within my replica's share of
    // the tile for the .ws layouts
    const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(lane_grp * 32) << 16) + static_cast<uint32_t>((WS ? u_local : u_begin) * kCols);
    // one register buffer: the load of unit r+1 is issued as soon as unit r has left the registers
    uint32_t vr[kCols];
    auto tmem_load = [&](int u) __attribute__((always_inline)) { ptx::tmem_ld16(taddr + u * kCols, vr); };
    tmem_load(0);
#pragma unroll
    for (int r = 0; r < kMaxUpw; ++r) {
      if (r < upw) {
        if (kHasRes && kPref < kMaxUpw && r > 0 && r % kPref == 0) prefetch_batch(r);  // next batch
        const int y = y_first + kUnitRows * r;  // first image row of the unit
        ptx::tmem_ld_wait();
        if (r < 2) MVLM_EPI_TRACE(8 + 4 * r);
        if (y < s.h) {
          if (F & F_HEAD) {
            // channel-major consumers: lane = channel c_lane, vr[j] = pixel (y + j/8, x0 + j%8)
            const int x0 = tc.tx * kTileW;
            const int nvx = s.w - x0;  // >= 8 for interior tiles
            // Arg-max only (the conv11 phase kernels, whose epilogue is their bound: ~130 instructions per unit for a
            // per-row tournament over ordered keys).  Most units cannot change the running maximum of their channel,
            // and those that can need the position of ONE value: a NaN-propagating 3-input max over the unit (+ bias:
            // the addition is monotonic, so max(v) + b == max(v + b) bit for bit) is compared with the running best
            // (">=": an equal value at a lower pixel index must still win, tiles are not visited in pixel order); only
            // then the first pixel whose biased value has exactly those bits is looked up.  A NaN in the unit takes the
            // exact per-row search below, which is also what the fp32-map variants run.
            bool exact_search = c_lane < e.cout_real;
            if constexpr ((F & F_HEAD) == F_ARGMAX) {
              if (c_lane < e.cout_real) {
                // two instantiations: every pixel of the unit exists (no masks at all) | edge tiles
                auto unit = [&](auto interior_c) __attribute__((always_inline)) {
                  constexpr bool kInterior = decltype(interior_c)::value;
                  auto ok = [&](int j) __attribute__((always_inline)) { return kInterior || ((j & 7) < nvx && y + (j >> 3) < s.h); };
                  float w[kCols];
#pragma unroll
                  for (int j = 0; j < kCols; ++j) w[j] = ok(j) ? __uint_as_float(vr[j]) : -INFINITY;
                  float m = fmax3_nan(w[0], w[1], w[2]);
#pragma unroll
                  for (int j = 3; j + 1 < kCols; j += 2) m = fmax3_nan(m, w[j], w[j + 1]);
                  m = fmax_nan(m, w[kCols - 1]);
                  const float mb = m + bias_c;
                  const uint32_t key = order_f32(mb);
                  exact_search = mb != mb;
                  if (key >= am.best_hi && !exact_search) {
                    const uint32_t mbits = __float_as_uint(mb);
                    int jf = kCols - 1;  // (masked pixels hold -inf: they must not stand in for a real -inf)
#pragma unroll
                    for (int j = kCols - 2; j >= 0; --j)
                      if (__float_as_uint(w[j] + bias_c) == mbits && ok(j)) jf = j;
                    const int oy = (y + (jf >> 3)) * e.up_sy + e.up_py;
                    const uint32_t lo = 0xFFFFFFFFu - static_cast<uint32_t>(oy * ow + (x0 + (jf & 7)) * e.up_sx + e.up_px);
                    if (key > am.best_hi || lo > am.best_lo) {
                      am.best_hi = key;
                      am.best_lo = lo;
                    }
                  }
                };
                if (nvx >= kTileW && y + kUnitRows <= s.h) unit(std::true_type());
                else unit(std::false_type());
              }
            }
            if (exact_search) {
#pragma unroll
              for (int i = 0; i < kUnitRows; ++i) {
                if (y + i < s.h) {
                  const int oy = (y + i) * e.up_sy + e.up_py;
                  const uint32_t idx0 = static_cast<uint32_t>(oy * ow + x0 * e.up_sx + e.up_px);
                  if (F & F_ARGMAX) {
                    // first maximum of the row's 8 pixels by a tournament over ordered keys (pixel index grows
                    // with j, so "the later one only if strictly greater" keeps the first), then ONE merge with
                    // the running best: a serial compare-select chain per pixel made this epilogue latency-bound
                    uint32_t k8[8];
                    uint32_t j8[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                      k8[j] = j < nvx ? order_f32(__uint_as_float(vr[8 * i + j]) + bias_c) : 0u;
                      j8[j] = static_cast<uint32_t>(j);
                    }
#pragma unroll
                    for (int st = 1; st < 8; st *= 2) {
#pragma unroll
                      for (int j = 0; j < 8; j += 2 * st) {
                        const bool take = k8[j + st] > k8[j];
                        k8[j] = take ? k8[j + st] : k8[j];
                        j8[j] = take ? j8[j + st] : j8[j];
                      }
                    }
                    const uint32_t lo = 0xFFFFFFFFu - (idx0 + j8[0] * static_cast<uint32_t>(e.up_sx));
                    if (k8[0] > am.best_hi || (k8[0] == am.best_hi && lo > am.best_lo)) {
                      am.best_hi = k8[0];
                      am.best_lo = lo;
                    }
                  }
                  if (F & F_F32) {
                    float* dst = e.out_f32 + (static_cast<size_t>(tc.img) * e.cout_real + c_lane) * oh * ow + idx0;
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                      if (j < nvx) dst[j * e.up_sx] = __uint_as_float(vr[8 * i + j]) + bias_c;
                  }
                }
              }
            }
          }
          if (kBf16Out) {
            // bias in the channel-major role (one register), then transpose the unit through shared memory:
            // row = pixel, 36 (20)-float pitch (conflict-free STS.32; LDS.128 conflict-free at 36)
            __syncwarp();
            {
#pragma unroll
              for (int j = 0; j < kCols; ++j) {
                float f = __uint_as_float(vr[j]) + bias_c;
                if (F & F_MID) f = fmaxf(fmaf(f, mid_s_c, mid_t_c), 0.f);
                stage[j * kPitch + lane] = f;
              }
            }
          }
        }
        if (r + 1 < upw) tmem_load(r + 1);  // next unit in flight while this one is post-processed
        if (y < s.h) {
          if (kBf16Out) {
            __syncwarp();
            if (r < 2) MVLM_EPI_TRACE(9 + 4 * r);
            uint4 pool_cur[2];
#pragma unroll
            for (int ip = 0; ip < 2; ++ip) {
              const int row = kUnitRows * r + ip;  // my image row in this pass, relative to my first
              const bool valid = row < n_rows_ok;
              float f[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
              if (valid) {
                lds8(stage + (pj + 8 * ip) * kPitch + cq, f);
                if (F & F_PRE)
                  *reinterpret_cast<uint4*>(b_pre + static_cast<size_t>(row * rs_pre)) = affine_relu_pack8(f, pre_s, pre_t);
                if (F & F_RES1) add8(r1[r % kPref][ip], f);
                if (F & F_RES2) add8(r2[r % kPref][ip], f);
                if (F & F_UP) add8(ru[r % kPref][0], f);
              }
              if (F & (F_POOL | F_POOLX)) pool_cur[ip] = pack8(f);
              if (!(F & F_POOL) && valid) {
                if (F & F_RAW) *reinterpret_cast<uint4*>(b_raw + static_cast<size_t>(row * rs_raw)) = (F & F_POOLX) ? pool_cur[ip] : pack8(f);
                if (F & F_POST)
                  *reinterpret_cast<uint4*>(b_post + static_cast<size_t>(row * rs_post)) = affine_relu_pack8(f, post_s, post_t);
                if (F & F_POST2) {
                  // parameters fetched from shared memory at the point of use: 16 registers this variant cannot hold
                  // across the tile
                  // (applied to the bf16-rounded raw value, like the stand-alone pass that reads the stored tensor)
                  float ax_s[8], ax_t[8], g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                  add8(pack8(f), g);
                  lds8(ep.mid_s + c0_ok, ax_s);
                  lds8(ep.mid_t + c0_ok, ax_t);
                  *reinterpret_cast<uint4*>(b_aux1 + static_cast<size_t>(row * rs_aux1)) = affine_relu_pack8(g, ax_s, ax_t);
                }
              }
            }
            if (r < 2) MVLM_EPI_TRACE(10 + 4 * r);
            if (F & (F_POOL | F_POOLX)) {
              // 2x2 max-pool of the bf16-rounded values; shuffles run on all lanes.  Vertical partner = my other
              // pass, horizontal (pixel column pj ^ 1) = lane ^ 4, one pooled row per unit.
              {
                uint4 m = max_bf16x8(pool_cur[0], pool_cur[1]);
                uint4 o;
                o.x = __shfl_xor_sync(0xffffffffu, m.x, 4);
                o.y = __shfl_xor_sync(0xffffffffu, m.y, 4);
                o.z = __shfl_xor_sync(0xffffffffu, m.z, 4);
                o.w = __shfl_xor_sync(0xffffffffu, m.w, 4);
                m = max_bf16x8(m, o);
                // H, W even: row y+1 and column xa+1 exist whenever (y, xa) does
                const int prow = r;  // pooled row relative to y_first / 2
                if (2 * prow < n_rows_ok && (pj & 1) == 0) {
                  if (F & F_POOL) {
                    if (F & F_RAW) *reinterpret_cast<uint4*>(b_raw + static_cast<size_t>(prow * rs_raw)) = m;
                    if (F & F_POST) {
                      float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                      add8(m, g);
                      *reinterpret_cast<uint4*>(b_post + static_cast<size_t>(prow * rs_post)) = affine_relu_pack8(g, post_s, post_t);
                    }
                  } else {  // F_POOLX: the pooled copies go to the aux tensors, raw / post were stored at full resolution
                    *reinterpret_cast<uint4*>(b_aux1 + static_cast<size_t>(prow * rs_aux1)) = m;
                    float g[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, ax_s[8], ax_t[8];
                    add8(m, g);
                    lds8(ep.mid_s + c0_ok, ax_s);
                    lds8(ep.mid_t + c0_ok, ax_t);
                    *reinterpret_cast<uint4*>(b_aux2 + static_cast<size_t>(prow * rs_aux2)) = affine_relu_pack8(g, ax_s, ax_t);
                  }
                }
              }
            }
            if (r < 2) MVLM_EPI_TRACE(11 + 4 * r);
          }
        }
      }
    }
  }
}

// flush of the running arg-max at the end of a CTA's tile range (arg-max convs have a single M tile)
template <int F>
__device__ __forceinline__ void epilogue_argmax_flush(const ConvShape& s, const ConvEpilogue& e, const int lane_grp,
                                                      const int lane, const ArgmaxState& am) {
  if ((F & F_ARGMAX) && am.cur_img >= 0 && am.best_hi != 0u) {
    constexpr bool WS = (F & F_M64) != 0;
    const int n_cgrp = !WS ? 4 : (s.cout_pad <= 32 ? 1 : 2);
    const int c_lane = (lane_grp & (n_cgrp - 1)) * 32 + lane;
    if (c_lane < e.cout_real)
      atomicMax(e.argmax_keys + static_cast<size_t>(am.cur_img) * e.cout_real + c_lane,
                (static_cast<unsigned long long>(am.best_hi) << 32) | am.best_lo);
  }
}

#endif  // __CUDACC__

}  // namespace epi
}  // namespace mvlm
