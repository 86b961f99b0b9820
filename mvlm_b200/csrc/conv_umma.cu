// tcgen05/TMEM implicit-GEMM convolution, see conv_umma.cuh for the contract.
//
// GEMM orientation ("weights are the A operand"):
//     D[cout (M=128 TMEM lanes) x pixels (N=256 TMEM columns)] += W[cout x K] * X[K x pixels]
// A single-CTA tcgen05.mma streams its A operand (128 rows x K=16) from shared memory at ~64 B/clk,
// i.e. >= ~75 cycles per instruction however small N is (measured: 79/84/94 cycles at N=32/64/128
// against a 16/32/64-cycle math floor).  With the 128 output channels as A and a whole 256-pixel
// tile as B (N=256) the same instruction does 128 cycles of math (measured 145), so the A stream is
// hidden -- see tools/exp_mma_only.py and DESIGN.md section 4.
//
// One persistent CTA per SM, 11 warps:
//   warp 0      TMA producer   X: ONE halo tile (8+KW-1 px x 32+KH-1 rows x 64 ch) per cin-chunk
//   warp 10     TMA producer   W: one [<=128 cout][64 cin] tile per (cin-chunk, kx, ky)
//   warp 1      MMA issuer     one elected lane issues tcgen05.mma (M=128, N=256, K=16); owns TMEM
//   warps 2..9  epilogue       tcgen05.ld (lane = channel, 16 pixels) -> smem transpose ->
//                              bias/BN/ReLU/residual on (pixel, 8 channels) vectors -> 16-byte stores
//
// Output tile = 8 px x 32 rows (N = 256; 16/8/4 rows for maps lower than 32).  The halo tile of a
// 64-channel chunk is stored pixel-major (128-byte rows, SWIZZLE_128B); the B operand of tap (kx, ky)
// is a descriptor into that SAME tile: start address shifted by (ky*(8+KW-1) + kx) rows of 128 bytes,
// stride between 8-row groups (SBO) = one halo row of (8+KW-1)*128 bytes.  Neither is a multiple of
// the 1024-byte swizzle atom: the hardware applies the swizzle XOR to the absolute shared-memory
// address (measured, tools/exp_swizzle_shift.cu: all taps / all swizzle widths bit-exact with base
// offset 0), so one TMA load serves all KW*KH taps -- 1.33x the tile's own pixels instead of 3.4x
// (one load per horizontal tap), which matters because the L2 -> SM fabric is the binding resource
// (10 TB/s on the 256->128 layers before this change).  Zero padding, ragged edges and maps smaller
// than the tile come from TMA out-of-bounds zero fill.
//
// Accumulators: 2 pipeline stages x 256 fp32 columns of TMEM: the epilogue of tile i overlaps the
// MMAs of tile i+1.
#include "conv_epilogue.cuh"

#include <algorithm>
#include <type_traits>
#include <atomic>

namespace mvlm {

namespace {

using namespace epi;
constexpr int kMaxHSlots = 4;                           // halo (activation) ring, depth chosen per layer
constexpr int kMaxWSlots = 12;                          // weight ring (16 KB slots at M = 128, 8 KB at M = 64)
constexpr int kPoolBytes = 198 * 1024;                  // both rings

struct __align__(8) Barriers {
  uint64_t h_full[kMaxHSlots];
  uint64_t h_empty[kMaxHSlots];
  uint64_t w_full[kMaxWSlots];
  uint64_t w_empty[kMaxWSlots];
  uint64_t t_full[2];
  uint64_t t_empty[2];
  uint32_t tmem_base;
};
static_assert(sizeof(Barriers) <= 512, "barrier block");

// Per-output-channel epilogue parameters staged once per CTA in shared memory.
struct EpiParams {
  float bias[kMaxCout];
  float mid_s[kMaxCout];
  float mid_t[kMaxCout];
  float pre_s[kMaxCout];
  float pre_t[kMaxCout];
  float post_s[kMaxCout];
  float post_t[kMaxCout];
};

constexpr int kSmemBytes = kPoolBytes + kEpiWarps * kStageFloats * 4 + 512 + static_cast<int>(sizeof(EpiParams)) +
                           1024 /*align*/;
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int t) {
  TileCoord c;
  c.mt = t % p.n_nt;
  int r = t / p.n_nt;
  c.tx = r % p.tiles_x;
  r /= p.tiles_x;
  c.ty = r % p.tiles_y;
  c.img = r / p.tiles_y;
  return c;
}

// Tile coordinates of a role's tile sequence t_begin, t_begin + t_step, ...: the three integer divisions are done once
// for the first tile and once for the step; every further tile is three additions with carry.  (Per tile they were a
// ~450-cycle dependent chain at the head of the epilogue warps' preamble, which the epilogue-bound layers pay in full.)
struct TileIter {
  TileCoord c, d;
  int n_nt, tiles_x, tiles_y;
  __device__ __forceinline__ TileIter(const ConvParams& p, int t_begin, int t_step)
      : c(decode_tile(p, t_begin)), d(decode_tile(p, t_step)), n_nt(p.n_nt), tiles_x(p.tiles_x), tiles_y(p.tiles_y) {}
  __device__ __forceinline__ void next() {
    c.mt += d.mt;
    int carry = c.mt >= n_nt ? 1 : 0;
    c.mt -= carry ? n_nt : 0;
    c.tx += d.tx + carry;
    carry = c.tx >= tiles_x ? 1 : 0;
    c.tx -= carry ? tiles_x : 0;
    c.ty += d.ty + carry;
    carry = c.ty >= tiles_y ? 1 : 0;
    c.ty -= carry ? tiles_y : 0;
    c.img += d.img + carry;
  }
};

template <int F>
__global__ void __launch_bounds__(kThreads, 1) conv_umma_kernel(const __grid_constant__ ConvParams p) {
  constexpr bool ARGMAX = (F & F_ARGMAX) != 0;  // arg-max variants use the contiguous tile schedule
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: TMA and UMMA agree on the SWIZZLE_128B XOR pattern through the absolute address
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* h_slots = smem;
  uint8_t* w_slots = smem + p.n_hslots * p.h_slot_bytes;
  float* stage_all = reinterpret_cast<float*>(smem + kPoolBytes);
  Barriers* bar = reinterpret_cast<Barriers*>(reinterpret_cast<uint8_t*>(stage_all) + kEpiWarps * kStageFloats * 4);
  EpiParams* ep = reinterpret_cast<EpiParams*>(reinterpret_cast<uint8_t*>(bar) + 512);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const ConvShape& s = p.s;
  const ConvEpilogue& e = p.e;
  const int n_chunks = (s.cin + 63) >> 6;
  const int n_hslots = p.n_hslots, n_wslots = p.n_wslots;
  const int halo_px = kTileW + s.kw - 1;            // pixels per halo row
  const int halo_rows = p.tile_h + s.kh - 1;
  // cout <= 64 runs with tcgen05.mma.ws, M = 64 (33 .. 64 channels) or 32: the plain M = 64 form leaves half of the
  // tensor core's 128 lanes idle (128.5 cycles per instruction at N = 256, like M = 128; tools/exp_m64.cu), the .ws
  // form spreads the 64 (32) x N tile over all 128 TMEM lanes and issues every 84.5 cycles (tools/exp_ws.cu), so
  // every epilogue warp holds 32 channels in its 32 lanes and the lane groups split the tile's pixel rows.
  constexpr bool M64 = (F & F_M64) != 0;
  constexpr bool STAT = (F & F_STAT) != 0;  // stationary weights and 3 x 3 (.ws) or 2 x 2 (M = 128) taps (conv_launch)
  constexpr int kM = M64 ? 64 : kMTile;
  const int w_rows = s.cout_pad < kM ? s.cout_pad : kM;  // weight rows actually loaded per tile
  const int mma_m = M64 ? (s.cout_pad <= 32 ? 32 : 64) : kMTile;
  // Weight ring.  M = 128: one slot = one (chunk, tap) tile of 16 KB.  .ws layers (M64): one slot = the KH taps of a
  // (chunk, kx) column, 8 KB apart (narrow tail chunks likewise): one barrier round trip per column -- per tap the
  // wait + commit + ring bookkeeping of the issuing thread take ~250-350 cycles (tools/exp_issue.cu), which 4 x 128
  // cycles of M = 128 math hide and 4 x 80 cycles of .ws math do not.
  // (M = 128 slots hold the rows that are loaded, rounded up to the 1 KB swizzle atom: 10 KB for the 80-channel heads.)
  const uint32_t w_tap_bytes = M64 ? 64u * 128u : ((static_cast<uint32_t>(w_rows) * 128u + 1023u) & ~1023u);  // tap stride inside a slot
  const uint32_t w_slot_bytes = w_tap_bytes * static_cast<uint32_t>(M64 ? s.kh : 1);
  // stationary weights: all (chunk, tap) tiles of the layer fit in the ring -> loaded once per CTA, never released
  const bool w_stat = p.w_stationary != 0;

  // Tile schedule shared by the three roles.  Default: round-robin (neighbouring CTAs work on neighbouring
  // tiles -> halo / weight reuse in L2).  ARGMAX: contiguous ranges, so that a CTA stays within one image
  // for ~40 tiles and keeps its running arg-max in registers.
  int t_begin, t_end, t_step;
  if (ARGMAX) {
    const int per = (p.total_tiles + gridDim.x - 1) / gridDim.x;
    t_begin = blockIdx.x * per;
    t_end = min(p.total_tiles, t_begin + per);
    t_step = 1;
  } else {
    t_begin = blockIdx.x; t_end = p.total_tiles; t_step = gridDim.x;
  }

  for (int i = threadIdx.x; i < s.cout_pad; i += kThreads) {
    ep->bias[i] = e.bias ? e.bias[i] : 0.f;
    ep->mid_s[i] = e.mid_scale ? e.mid_scale[i] : (e.aux_scale ? e.aux_scale[i] : 1.f);  // aux parameters share the slot
    ep->mid_t[i] = e.mid_scale ? e.mid_shift[i] : (e.aux_shift ? e.aux_shift[i] : 0.f);
    ep->pre_s[i] = e.out_pre ? e.pre_scale[i] : 0.f;
    ep->pre_t[i] = e.out_pre ? e.pre_shift[i] : 0.f;
    ep->post_s[i] = e.out_post ? e.post_scale[i] : 0.f;
    ep->post_t[i] = e.out_post ? e.post_shift[i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    ptx::tma_prefetch_desc(&p.tm_a);
    ptx::tma_prefetch_desc(&p.tm_b);
    if (p.tail) { ptx::tma_prefetch_desc(&p.tm_a2); ptx::tma_prefetch_desc(&p.tm_b2); }
    if (F & F_RES1) ptx::tma_prefetch_desc(&p.tm_r1);
    if (F & F_RES2) ptx::tma_prefetch_desc(&p.tm_r2);
    if (F & F_UP) ptx::tma_prefetch_desc(&p.tm_up);
    for (int i = 0; i < n_hslots; ++i) {
      ptx::mbar_init(&bar->h_full[i], 1);
      ptx::mbar_init(&bar->h_empty[i], 1);
    }
    for (int i = 0; i < n_wslots; ++i) {
      ptx::mbar_init(&bar->w_full[i], 1);
      ptx::mbar_init(&bar->w_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&bar->t_full[i], 1);
      ptx::mbar_init(&bar->t_empty[i], kEpiWarps);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 1) {
    ptx::tmem_alloc(&bar->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  // Programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch, per-channel parameters,
  // none of which another launch of the plan writes) may overlap the tail of the previous kernel in the stream;
  // every read or write of an activation tensor comes after this wait.  The next kernel may start its own
  // prologue as soon as SMs free up.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t tmem_base = bar->tmem_base;
  const bool prof = p.prof != nullptr;
  const long long t_kernel0 = clock64();
  long long w0 = 0, w1 = 0;
  // per-tile timeline of CTA 0 (first kTraceTiles tiles), cycles since kernel start:
  //   [0] producer: halo load of chunk 0 issued   [1] producer: last weight load issued
  //   [2] MMA: accumulator stage acquired         [3] MMA: first halo tile landed      [4] MMA: all MMAs issued
  //   [5] epilogue warp 2: accumulator ready      [6] epilogue warp 2: stage released
  //   epilogue warp 2, unit r = 0 / 1: [8 + 4r] accumulator columns in registers, [9 + 4r] transposed to shared
  //   memory, [10 + 4r] outputs computed and stores issued, [11 + 4r] unit done (rolling prefetch issued)
  long long* const trace = (prof && blockIdx.x == 0) ? p.prof + kNumSMs * 8 : nullptr;
  int trace_i = 0;
#define MVLM_TRACE(slot)                                                                  \
  do {                                                                                    \
    if (trace && trace_i < kTraceTiles) trace[trace_i * 16 + (slot)] = clock64() - t_kernel0; \
  } while (0)

  if (warp == 0) {
    // ===================== TMA producer: activations =====================
    // Its own thread, so that the halo prefetch runs n_hslots chunks ahead of the MMAs whatever the state of the
    // weight ring (measured: behind the weight loads in one queue the next halo tile was issued ~4k cycles before
    // it was needed, about the DRAM + queueing latency of the load, and the tensor pipe waited for it every tile).
    if (ptx::elect_one() && (p.debug_mode & 1) == 0) {
      int sh = 0;
      uint32_t ph = 0;
      TileIter it(p, t_begin, t_step);
      for (int t = t_begin; t < t_end; t += t_step, it.next()) {
        const TileCoord tc = it.c;
        const int x0 = tc.tx * kTileW + s.x_off0;
        const int y0 = tc.ty * p.tile_h + s.y_off0;
        for (int c = 0; c < n_chunks; ++c) {
          // the last chunk may be a narrow tail (16 / 32 channels) with its own tensor map: rows of 32 / 64 bytes
          const bool is_tail = p.tail != 0 && c == n_chunks - 1;
          const uint32_t row_b = is_tail ? static_cast<uint32_t>(p.tail) * 2u : 128u;  // bytes per pixel
          timed_wait(&bar->h_empty[sh], ph ^ 1, prof, w0);
          ptx::mbar_expect_tx(&bar->h_full[sh], static_cast<uint32_t>(halo_rows * halo_px) * row_b);
          // one halo tile for all KW x KH taps of this chunk
          ptx::tma_load_4d(is_tail ? &p.tm_a2 : &p.tm_a, &bar->h_full[sh], h_slots + sh * p.h_slot_bytes, c * 64, x0, y0, tc.img);
          if (c == 0) MVLM_TRACE(0);
          if (++sh == n_hslots) { sh = 0; ph ^= 1; }
        }
        // Residual inputs of this tile -> L2, now, i.e. one to two tiles before the epilogue warps load them: this
        // thread is idle between halo loads, the epilogue warps are not (their loads for a tile are issued ~1.5k
        // cycles before the first use, DRAM latency under load is ~2.5k: the first unit of every tile waited 1.9k
        // cycles on the 256^2 64->64 layer).  One TMA box per residual tensor (per-pixel bulk prefetches made this
        // thread the bottleneck: ~35 cycles each).
        if constexpr ((F & (F_RES1 | F_RES2 | F_UP)) != 0) {
          const int xa = tc.tx * kTileW, ya = tc.ty * p.tile_h, c_lo = tc.mt * kM;
          if (F & F_RES1) ptx::tma_prefetch_l2_4d(&p.tm_r1, c_lo, xa, ya, tc.img);
          if (F & F_RES2) ptx::tma_prefetch_l2_4d(&p.tm_r2, c_lo, xa, ya, tc.img);
          if (F & F_UP) ptx::tma_prefetch_l2_4d(&p.tm_up, c_lo, xa >> 1, ya >> 1, tc.img);
        }
        ++trace_i;
      }
      if (prof) { p.prof[blockIdx.x * 8 + 0] = w0; p.prof[blockIdx.x * 8 + 7] = clock64() - t_kernel0; }
    }
  } else if (warp == 10) {
    // ===================== TMA producer: weights =====================
    if (ptx::elect_one() && (p.debug_mode & 1) == 0) {
      int sw = 0;
      uint32_t pw = 0;
      for (int t = t_begin; t < t_end; t += t_step) {
        const int mt = t % p.n_nt;
        for (int c = 0; c < n_chunks; ++c) {
          const bool is_tail = p.tail != 0 && c == n_chunks - 1;
          const void* tmb = is_tail ? &p.tm_b2 : &p.tm_b;
          const uint32_t row_b = is_tail ? static_cast<uint32_t>(p.tail) * 2u : 128u;  // bytes per weight row
          const uint32_t wb = static_cast<uint32_t>(w_rows) * row_b;
          if constexpr (M64) {
            for (int kx = 0; kx < s.kw; ++kx) {  // one slot per column of taps (tap = kx * KH + ky)
              if (!w_stat) timed_wait(&bar->w_empty[sw], pw ^ 1, prof, w1);
              ptx::mbar_expect_tx(&bar->w_full[sw], wb * static_cast<uint32_t>(s.kh));
              for (int ky = 0; ky < s.kh; ++ky)
                ptx::tma_load_2d(tmb, &bar->w_full[sw], w_slots + sw * w_slot_bytes + ky * w_tap_bytes,
                                 (kx * s.kh + ky) * s.cin + c * 64, mt * kM);
              if (++sw == n_wslots) { sw = 0; pw ^= 1; }
            }
          } else
          for (int tap = 0; tap < s.kw * s.kh; ++tap) {  // tap = kx * KH + ky
            if (!w_stat) timed_wait(&bar->w_empty[sw], pw ^ 1, prof, w1);
            ptx::mbar_expect_tx(&bar->w_full[sw], wb);
            ptx::tma_load_2d(tmb, &bar->w_full[sw], w_slots + sw * w_slot_bytes, tap * s.cin + c * 64, mt * kM);
            if (++sw == n_wslots) { sw = 0; pw ^= 1; }
          }
        }
        MVLM_TRACE(1);
        ++trace_i;
        if (w_stat) break;  // one pass over the layer's weights is all there is
      }
      if (prof) p.prof[blockIdx.x * 8 + 1] = w1;
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // elect.sync (not `lane == 0`): the compiler then knows a single lane is active and emits the
    // UTCHMMA / UTCBAR uniform-datapath instructions without a per-lane serialisation loop.
    if (ptx::elect_one()) {
      // This loop is ONE thread's dependent scalar code: with ~80 instructions per tap (barrier bookkeeping, constant-bank
      // reloads, descriptor arithmetic) it took ~450 cycles per tap whatever the number of MMAs in it (measured with
      // operands and epilogue switched off, tools/exp_ws_inkernel.py) -- hidden behind 4 x 128 cycles of math at M = 128,
      // not behind 4 (2, 1) x 80 cycles of the .ws layers.  So: everything that does not change per tap is hoisted, the
      // descriptors advance by integer adds, stationary weights are waited for once per CTA, and there is no
      // tcgen05.fence in the tap loop (the mbarrier wait orders the TMA writes before the MMA's reads).
      const uint32_t idesc = ptx::umma_idesc_bf16(mma_m, p.tile_h * kTileW);
      // descriptor = {lo: start>>4 | LBO, hi: SBO | version | swizzle}; only lo changes per MMA.
      //   A (weights): 8-row groups 8 rows apart.  B (halo tile): 8-row group = the 8 pixels of one image row,
      //   groups one halo row (halo_px pixels) apart.
      // full 64-channel chunks: 128-byte rows, SWIZZLE_128B; tail chunk: SWIZZLE_32B (16 ch: 32-byte rows) or
      // SWIZZLE_64B (32 ch: 64-byte rows)
      const bool live = (p.debug_mode & 1) == 0;
      const int n_kx = s.kw, n_ky = s.kh;
      const uint32_t tail_row_b = p.tail ? static_cast<uint32_t>(p.tail) * 2u : 128u;
      const uint32_t tail_swz = !p.tail ? 2u : (p.tail == 16 ? 6u : 4u);
      const uint64_t a_hi_full = static_cast<uint64_t>(((8u * 128u) >> 4) | (1u << 14) | (2u << 29)) << 32;
      const uint64_t b_hi_full = static_cast<uint64_t>(((static_cast<uint32_t>(halo_px) * 128u) >> 4) | (1u << 14) | (2u << 29)) << 32;
      const uint64_t a_hi_tail = static_cast<uint64_t>(((8u * tail_row_b) >> 4) | (1u << 14) | (tail_swz << 29)) << 32;
      const uint64_t b_hi_tail = static_cast<uint64_t>(((static_cast<uint32_t>(halo_px) * tail_row_b) >> 4) | (1u << 14) | (tail_swz << 29)) << 32;
      // shared-memory addresses are below 2^18: (address >> 4) needs no mask and slot offsets are plain adds
      const uint32_t h_lo0 = (ptx::smem_u32(h_slots) >> 4) | (1u << 16), h_step = static_cast<uint32_t>(p.h_slot_bytes) >> 4;
      const uint32_t w_lo0 = (ptx::smem_u32(w_slots) >> 4) | (1u << 16), w_step = w_slot_bytes >> 4;
      const int last_chunk = n_chunks - 1;
      const int nk_last = (s.cin - last_chunk * 64) >= 64 ? 4 : ((s.cin - last_chunk * 64) >> 4);
      int sh = 0, sw = 0;
      uint32_t ph = 0, pw = 0;
      int acc = 0;
      uint32_t pacc = 0;
      bool w_wait = live;  // stationary weights: the slots are waited for during the first tile only
      for (int t = t_begin; t < t_end; t += t_step) {
        timed_wait(&bar->t_empty[acc], pacc ^ 1, prof, w1);
        ptx::tc_fence_after();
        MVLM_TRACE(2);
        const uint32_t d = tmem_base + static_cast<uint32_t>(acc * 256);
        uint32_t accumulate = 0;
        for (int c = 0; c < n_chunks; ++c) {
          const bool is_tail = p.tail != 0 && c == last_chunk;
          const int nk = c == last_chunk ? nk_last : 4;
          const uint32_t rb16 = (is_tail ? tail_row_b : 128u) >> 4;  // 16-byte units per pixel row
          const uint64_t a_hi = is_tail ? a_hi_tail : a_hi_full;
          const uint64_t b_hi = is_tail ? b_hi_tail : b_hi_full;
          const uint32_t ky_step = static_cast<uint32_t>(halo_px) * rb16;
          if (live) timed_wait(&bar->h_full[sh], ph, prof, w0);
          if (c == 0) MVLM_TRACE(3);
          uint32_t x_col = h_lo0 + static_cast<uint32_t>(sh) * h_step;
          if (STAT && !w_wait && (nk == 4 || nk == 2 || nk == 1)) {
            // Stationary weights that have been waited for, 3 x 3 (.ws layers) or 2 x 2 taps (the conv11 phase kernels),
            // straight-line: the B descriptor of tap (kx, ky), K-step k is x_col + a compile-time offset (halo rows are
            // 8 + KW - 1 pixels of NK * 32 bytes), the A descriptor is tile chunk * taps + tap: two uniform adds per MMA,
            // no barrier in sight.  (The same unrolling with the weight ring's wait / commit per tap made the 128- and
            // 256-channel layers 3-4 % slower.)
            auto taps = [&](auto nk_c, auto kk_c) __attribute__((always_inline)) {
              constexpr int NK = decltype(nk_c)::value;
              constexpr int KK = decltype(kk_c)::value;  // KW = KH
              constexpr uint32_t kRb16 = NK * 2;
              const uint32_t tap16 = M64 ? (64u * 128u >> 4) : w_step;  // tap stride: 8 KB inside a column slot | one slot
              const uint32_t w_base = w_lo0 + static_cast<uint32_t>(c * KK * KK) * tap16;
#pragma unroll
              for (int tap = 0; tap < KK * KK; ++tap) {  // tap = kx * KH + ky
                const uint32_t x_lo = x_col + static_cast<uint32_t>(((tap % KK) * (kTileW + KK - 1) + tap / KK)) * kRb16;
                const uint32_t w_lo = w_base + static_cast<uint32_t>(tap) * tap16;
#pragma unroll
                for (int k = 0; k < NK; ++k) {
                  const uint32_t en = (tap == 0 && k == 0) ? accumulate : 1u;
                  if constexpr (M64) ptx::umma_ws_bf16(d, a_hi | (w_lo + 2 * k), b_hi | (x_lo + 2 * k), idesc, en);
                  else ptx::umma_bf16(d, a_hi | (w_lo + 2 * k), b_hi | (x_lo + 2 * k), idesc, en);
                }
              }
              accumulate = 1;
            };
            using std::integral_constant;
            if constexpr (M64) {
              if (nk == 4) taps(integral_constant<int, 4>(), integral_constant<int, 3>());
              else if (nk == 2) taps(integral_constant<int, 2>(), integral_constant<int, 3>());
              else taps(integral_constant<int, 1>(), integral_constant<int, 3>());
            } else {
              if (nk == 4) taps(integral_constant<int, 4>(), integral_constant<int, 2>());
              else if (nk == 2) taps(integral_constant<int, 2>(), integral_constant<int, 2>());
              else taps(integral_constant<int, 1>(), integral_constant<int, 2>());
            }
          } else if constexpr (M64) {
            // .ws layers: one ring slot per column of taps
            for (int kx = 0; kx < n_kx; ++kx, x_col += rb16) {
              if (w_wait) timed_wait(&bar->w_full[sw], w_stat ? 0u : pw, prof, w0);
              uint32_t x_lo = x_col;
              uint32_t w_lo = w_lo0 + static_cast<uint32_t>(sw) * w_step;
              for (int ky = 0; ky < n_ky; ++ky, x_lo += ky_step, w_lo += (w_tap_bytes >> 4)) {
                ptx::umma_ws_bf16(d, a_hi | w_lo, b_hi | x_lo, idesc, accumulate);
                if (nk == 4) {
                  ptx::umma_ws_bf16(d, a_hi | (w_lo + 2), b_hi | (x_lo + 2), idesc, 1u);
                  ptx::umma_ws_bf16(d, a_hi | (w_lo + 4), b_hi | (x_lo + 4), idesc, 1u);
                  ptx::umma_ws_bf16(d, a_hi | (w_lo + 6), b_hi | (x_lo + 6), idesc, 1u);
                } else {
                  for (int k = 1; k < nk; ++k) ptx::umma_ws_bf16(d, a_hi | (w_lo + 2 * k), b_hi | (x_lo + 2 * k), idesc, 1u);
                }
                accumulate = 1;
              }
              if (live && !w_stat) ptx::umma_commit(&bar->w_empty[sw]);
              if (++sw == n_wslots) { sw = 0; pw ^= 1; }
            }
          } else
          for (int kx = 0; kx < n_kx; ++kx, x_col += rb16) {
            // tap (kx, ky) = the same halo tile shifted by ky halo rows + kx pixels
            uint32_t x_lo = x_col;
            for (int ky = 0; ky < n_ky; ++ky, x_lo += ky_step) {
              if (w_wait) timed_wait(&bar->w_full[sw], w_stat ? 0u : pw, prof, w0);
              const uint32_t w_lo = w_lo0 + static_cast<uint32_t>(sw) * w_step;
              auto mma = [&](int k, uint32_t en) __attribute__((always_inline)) {
                if constexpr (M64) ptx::umma_ws_bf16(d, a_hi | (w_lo + 2 * k), b_hi | (x_lo + 2 * k), idesc, en);
                else ptx::umma_bf16(d, a_hi | (w_lo + 2 * k), b_hi | (x_lo + 2 * k), idesc, en);
              };
              mma(0, accumulate);
              if (nk == 4) {
                mma(1, 1u); mma(2, 1u); mma(3, 1u);
              } else {
                for (int k = 1; k < nk; ++k) mma(k, 1u);
              }
              accumulate = 1;
              if (live && !w_stat) ptx::umma_commit(&bar->w_empty[sw]);
              if (++sw == n_wslots) { sw = 0; pw ^= 1; }
            }
          }
          if (live) ptx::umma_commit(&bar->h_empty[sh]);
          if (++sh == n_hslots) { sh = 0; ph ^= 1; }
        }
        ptx::umma_commit(&bar->t_full[acc]);
        MVLM_TRACE(4);
        ++trace_i;
        if (w_stat) w_wait = false;
        if (++acc == 2) { acc = 0; pacc ^= 1; }
      }
      if (prof) { p.prof[blockIdx.x * 8 + 2] = w0; p.prof[blockIdx.x * 8 + 3] = w1; p.prof[blockIdx.x * 8 + 4] = clock64() - t_kernel0; }
    }
  } else {
    // ===================== epilogue =====================
    // the per-tile work is epi::epilogue_tile (conv_epilogue.cuh)
    float* stage = stage_all + (warp - 2) * kStageFloats;
    const ChannelParams cp = {ep->bias, ep->mid_s, ep->mid_t, ep->pre_s, ep->pre_t, ep->post_s, ep->post_t};
    int acc = 0;
    uint32_t pacc = 0;
    ArgmaxState am;
    EpiTrace tr;
    tr.trace = trace; tr.t0 = t_kernel0; tr.on = warp == 2 && lane == 0;
    TileIter it(p, t_begin, t_step);
    for (int t = t_begin; t < t_end; t += t_step, it.next()) {
      const TileCoord tc = it.c;
      tr.trace_i = trace_i;
      if (p.debug_mode & 2) {  // experiment: accumulators are dropped (results invalid)
        timed_wait(&bar->t_full[acc], pacc, prof, w0);
        ptx::tc_fence_after();
      } else {
        epilogue_tile<F>(s, e, p.tile_h, cp, tc, &bar->t_full[acc], pacc, tmem_base + static_cast<uint32_t>(acc * 256),
                         stage, warp - 2, warp & 3, lane, am, prof, w0, tr);
      }
      // all tcgen05.ld of this accumulator stage have completed (wait::ld above)
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&bar->t_empty[acc]);
      if (warp == 2 && lane == 0) MVLM_TRACE(6);
      ++trace_i;
      if (++acc == 2) { acc = 0; pacc ^= 1; }
    }
    epilogue_argmax_flush<F>(s, e, warp & 3, lane, am);
    if (prof && warp == 2 && lane == 0) { p.prof[blockIdx.x * 8 + 5] = w0; p.prof[blockIdx.x * 8 + 6] = clock64() - t_kernel0; }
  }

#undef MVLM_TRACE
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, 512);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* sym = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) != cudaSuccess ||
      q != cudaDriverEntryPointSuccess || !sym)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(sym);
  return fn;
}

template <int F>
int launch_t(const ConvParams& p, cudaStream_t stream) {
  // the attribute is per device (and per kernel instantiation): one flag per device ordinal
  static std::atomic<bool> configured[kMaxDevices];
  int dev = 0;
  MVLM_CHECK_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= kMaxDevices || !configured[dev].load(std::memory_order_acquire)) {
    MVLM_CHECK_CUDA(cudaFuncSetAttribute(conv_umma_kernel<F>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    if (dev >= 0 && dev < kMaxDevices) configured[dev].store(true, std::memory_order_release);
  }
  const int n_sms = sm_count();
  const int grid = p.total_tiles < n_sms ? p.total_tiles : n_sms;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemBytes;
  cfg.stream = stream;
  // programmatic dependent launch of consecutive conv kernels
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MVLM_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_umma_kernel<F>, p));
  count_launch();
  MVLM_CHECK_CUDA(cudaGetLastError());
  return MVLM_OK;
}

// debug hooks: set and read on the thread that profiles (thread-local: other threads' launches are unaffected)
thread_local long long* g_prof_buf = nullptr;
thread_local int g_debug_mode = 0;

}  // namespace

int conv_plan(const ConvShape& s, const ConvEpilogue& e, ConvParams* out) {
  MVLM_REQUIRE(s.in && s.wpacked, "conv_plan: null input/weights");
  MVLM_REQUIRE(s.n > 0 && s.h > 0 && s.w > 0, "conv_plan: bad image dims %d %d %d", s.n, s.h, s.w);
  MVLM_REQUIRE(s.cin >= 16 && s.cin % 16 == 0, "conv_plan: cin=%d must be a multiple of 16", s.cin);
  MVLM_REQUIRE(s.in_cs >= s.cin && s.in_cs % 8 == 0, "conv_plan: in_cs=%d invalid", s.in_cs);
  MVLM_REQUIRE(s.cout_pad >= 16 && s.cout_pad % 16 == 0, "conv_plan: cout_pad=%d must be a multiple of 16", s.cout_pad);
  MVLM_REQUIRE(s.cout_pad <= kMTile || s.cout_pad % kMTile == 0,
               "conv_plan: cout_pad=%d must be <= 128 or a multiple of 128", s.cout_pad);
  MVLM_REQUIRE(s.cout_pad <= kMaxCout, "conv_plan: cout_pad=%d exceeds %d", s.cout_pad, kMaxCout);
  MVLM_REQUIRE(!e.argmax_keys || s.cout_pad <= kMTile, "conv_plan: fused arg-max needs cout_pad <= 128");
  MVLM_REQUIRE(!e.pool2 || (s.h % 2 == 0 && s.w % 2 == 0 && (e.out_raw || e.out_post) && !e.out_f32 && !e.argmax_keys),
               "conv_plan: pool2 needs even H, W and a bf16 raw/post output");
  MVLM_REQUIRE(!e.res_up || (s.h % 2 == 0 && s.w % 2 == 0 && !e.pool2 && !e.out_f32 && !e.argmax_keys),
               "conv_plan: res_up needs even H, W and bf16 outputs");
  MVLM_REQUIRE(!e.mid_scale || (e.mid_shift && !e.out_f32 && !e.argmax_keys), "conv_plan: mid affine needs mid_shift and bf16 outputs");
  MVLM_REQUIRE(e.aux_mode >= 0 && e.aux_mode <= 2, "conv_plan: unknown aux_mode %d", e.aux_mode);
  MVLM_REQUIRE(e.aux_mode == 0 || (e.aux_scale && e.aux_shift && e.out_aux1 && !e.mid_scale && !e.pool2 && !e.out_f32 &&
                                   !e.argmax_keys && e.aux1_cs % 8 == 0),
               "conv_plan: aux copies need aux_scale / aux_shift / out_aux1 and cannot be combined with mid / pool2 / fp32 outputs");
  MVLM_REQUIRE(e.aux_mode != 2 || (e.out_aux2 && e.aux2_cs % 8 == 0 && s.h % 2 == 0 && s.w % 2 == 0),
               "conv_plan: pooled aux copies need out_aux2 and even H, W");
  MVLM_REQUIRE(!((e.argmax_keys || e.out_f32) && (e.res1 || e.res2 || e.out_pre || e.out_raw || e.out_post)),
               "conv_plan: fp32 / arg-max outputs cannot be combined with bf16 outputs or residual inputs");
  // pixel indices are 32-bit (they are widened before the multiplication with a channel stride)
  MVLM_REQUIRE(1ll * s.n * s.h * s.w < (1ll << 32), "conv_plan: %d x %d x %d pixels exceed 32-bit pixel indices", s.n, s.h, s.w);
  MVLM_REQUIRE(s.kh >= 1 && s.kh <= 3 && s.kw >= 1 && s.kw <= 3, "conv_plan: kernel %dx%d unsupported", s.kh, s.kw);
  MVLM_REQUIRE((reinterpret_cast<uintptr_t>(s.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(s.wpacked) & 15) == 0,
               "conv_plan: pointers must be 16-byte aligned");
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) {
    set_error("conv_plan: cuTensorMapEncodeTiled entry point unavailable");
    return MVLM_E_CUDA;
  }
  ConvParams p;
  memset(&p, 0, sizeof(p));
  p.s = s;
  p.e = e;
  // output tile: 8 px x tile_h rows (N = 8 * tile_h columns), tile_h = 32 unless the map is lower; the .ws MMA of the
  // cout <= 64 layers needs N >= 64 (rows beyond the map are TMA zero fill and never stored)
  const int tile_h = s.h >= 32 ? kMaxTileH : (s.h >= 16 ? 16 : ((s.h >= 8 || s.cout_pad <= 64) ? 8 : 4));
  p.tile_h = tile_h;
  {
    // ring depths: the halo slot holds the whole (8+KW-1) x (tile_h+KH-1) pixel tile of one 64-channel chunk
    const int hbytes = (kTileW + s.kw - 1) * (tile_h + s.kh - 1) * 128;
    p.h_slot_bytes = (hbytes + 1023) & ~1023;
    // cout <= 64 -> tcgen05.mma.ws with M <= 64, 8 KB weight slots; all (chunk, tap) tiles resident when they fit the ring
    const int m_tile = s.cout_pad <= 64 ? 64 : kMTile;
    // ring slot: the KH taps of one (chunk, kx) column for the .ws layers, one tap otherwise (see the kernel)
    const int w_tap = m_tile == 64 ? 64 * 128 : ((std::min(s.cout_pad, kMTile) * 128 + 1023) & ~1023);
    const int wslot = w_tap * (m_tile == 64 ? s.kh : 1);
    const int n_wtiles = ((s.cin + 63) / 64) * (m_tile == 64 ? s.kw : s.kh * s.kw);  // slots of one pass over the layer
    int nh = s.kh * s.kw == 1 ? 3 : 2, nw = s.kh * s.kw == 1 ? 6 : (m_tile == 64 ? kMaxWSlots : 7);
    // stationary weights: every slot of the layer resident (loaded once per CTA, no barrier traffic afterwards) -- the
    // .ws layers up to K = 768, and single-M-tile M = 128 layers whose weights fit next to the halo ring (the four
    // conv11 phase kernels: 8 x 10 KB; the 64 -> 128 resample)
    const bool fits_128 = m_tile == kMTile && s.cout_pad <= kMTile && n_wtiles <= kMaxWSlots &&
                          nh * p.h_slot_bytes + n_wtiles * wslot <= kPoolBytes;
    p.w_stationary = (m_tile == 64 ? n_wtiles * wslot <= kMaxWSlots * 8192 : fits_128) ? 1 : 0;
    if (p.w_stationary) nw = n_wtiles;
    while (nh * p.h_slot_bytes + nw * wslot > kPoolBytes && nw > 2 && !p.w_stationary) --nw;
    while (nh * p.h_slot_bytes + nw * wslot > kPoolBytes && nh > 2) --nh;
    MVLM_REQUIRE(nh * p.h_slot_bytes + nw * wslot <= kPoolBytes, "conv_plan: operand rings do not fit");
    p.n_hslots = nh;
    p.n_wslots = nw;
  }
  {
    // X: (C, W, H, N) bf16, box (64, 8+KW-1, tile_h+KH-1, 1), 128-byte swizzle, OOB -> 0
    cuuint64_t gdim[4] = {(cuuint64_t)s.cin, (cuuint64_t)s.w, (cuuint64_t)s.h, (cuuint64_t)s.n};
    cuuint64_t gstr[3] = {(cuuint64_t)s.in_cs * 2, (cuuint64_t)s.in_cs * 2 * s.w,
                          (cuuint64_t)s.in_cs * 2 * s.w * s.h};
    cuuint32_t box[4] = {64, (cuuint32_t)(kTileW + s.kw - 1), (cuuint32_t)(tile_h + s.kh - 1), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&p.tm_a, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(s.in), gdim, gstr,
                     box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("conv_plan: cuTensorMapEncodeTiled(X) failed with %d (cin=%d w=%d h=%d n=%d cs=%d)", (int)r, s.cin,
                s.w, s.h, s.n, s.in_cs);
      return MVLM_E_CUDA;
    }
  }
  {
    // W: (K = KW*KH*cin, cout_pad) bf16, box (64, min(cout_pad,128))
    const cuuint64_t ktot = (cuuint64_t)s.kw * s.kh * s.cin;
    cuuint64_t gdim[2] = {ktot, (cuuint64_t)s.cout_pad};
    cuuint64_t gstr[1] = {ktot * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)(s.cout_pad < kMTile ? s.cout_pad : kMTile)};  // cout_pad <= 64: M = 64 tile
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&p.tm_b, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(s.wpacked), gdim,
                     gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                     CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      set_error("conv_plan: cuTensorMapEncodeTiled(W) failed with %d (ktot=%llu cout_pad=%d)", (int)r,
                (unsigned long long)ktot, s.cout_pad);
      return MVLM_E_CUDA;
    }
  }
  p.tail = (s.cin % 64 == 16 || s.cin % 64 == 32) ? s.cin % 64 : 0;
  if (p.tail) {
    const CUtensorMapSwizzle sw = p.tail == 16 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B;
    cuuint64_t gdim[4] = {(cuuint64_t)s.cin, (cuuint64_t)s.w, (cuuint64_t)s.h, (cuuint64_t)s.n};
    cuuint64_t gstr[3] = {(cuuint64_t)s.in_cs * 2, (cuuint64_t)s.in_cs * 2 * s.w, (cuuint64_t)s.in_cs * 2 * s.w * s.h};
    cuuint32_t box[4] = {(cuuint32_t)p.tail, (cuuint32_t)(kTileW + s.kw - 1), (cuuint32_t)(tile_h + s.kh - 1), 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&p.tm_a2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(s.in), gdim, gstr, box,
                     estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    const cuuint64_t ktot = (cuuint64_t)s.kw * s.kh * s.cin;
    cuuint64_t gdim2[2] = {ktot, (cuuint64_t)s.cout_pad};
    cuuint64_t gstr2[1] = {ktot * 2};
    cuuint32_t box2[2] = {(cuuint32_t)p.tail, (cuuint32_t)(s.cout_pad < kMTile ? s.cout_pad : kMTile)};
    CUresult r2 = enc(&p.tm_b2, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(s.wpacked), gdim2,
                      gstr2, box2, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS || r2 != CUDA_SUCCESS) {
      set_error("conv_plan: cuTensorMapEncodeTiled(tail %d) failed with %d / %d", p.tail, (int)r, (int)r2);
      return MVLM_E_CUDA;
    }
  }
  {
    // residual inputs: (channel slice of cout_pad, W, H, N) from the slice's first channel; box = one output tile
    // (half of it for the half-resolution up-sample input), prefetch only -> no swizzle
    auto res_map = [&](CUtensorMap* tm, const __nv_bfloat16* base, int co, int cs, int hh, int ww, int box_w, int box_h) -> bool {
      if (!base) return true;
      const int c_ext = std::min(s.cout_pad, cs);  // the slice never extends past the pixel's channels
      cuuint64_t gdim[4] = {(cuuint64_t)c_ext, (cuuint64_t)ww, (cuuint64_t)hh, (cuuint64_t)s.n};
      cuuint64_t gstr[3] = {(cuuint64_t)cs * 2, (cuuint64_t)cs * 2 * ww, (cuuint64_t)cs * 2 * ww * hh};
      cuuint32_t box[4] = {(cuuint32_t)std::min(c_ext, s.cout_pad <= 64 ? 64 : kMTile), (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
      cuuint32_t estr[4] = {1, 1, 1, 1};
      return enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<__nv_bfloat16*>(base + co), gdim, gstr, box, estr,
                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    };
    const bool ok = res_map(&p.tm_r1, e.res1, e.res1_co, e.res1_cs, s.h, s.w, kTileW, tile_h) &&
                    res_map(&p.tm_r2, e.res2, e.res2_co, e.res2_cs, s.h, s.w, kTileW, tile_h) &&
                    res_map(&p.tm_up, e.res_up, e.up_co, e.up_cs, s.h >> 1, s.w >> 1, kTileW / 2, std::max(1, tile_h / 2));
    if (!ok) {
      set_error("conv_plan: cuTensorMapEncodeTiled(residual) failed (cout_pad=%d w=%d h=%d)", s.cout_pad, s.w, s.h);
      return MVLM_E_CUDA;
    }
  }
  p.tiles_x = ceil_div(s.w, kTileW);
  p.tiles_y = ceil_div(s.h, tile_h);
  p.n_nt = s.cout_pad <= 64 ? 1 : ceil_div(s.cout_pad, kMTile);
  p.total_tiles = s.n * p.tiles_x * p.tiles_y * p.n_nt;
  p.prof = nullptr;
  p.debug_mode = 0;
  *out = p;
  return MVLM_OK;
}

void conv_set_profile_buffer(long long* dev_buf) { g_prof_buf = dev_buf; }
void conv_set_debug_mode(int mode) { g_debug_mode = mode; }

int conv_launch(const ConvParams& p_in, cudaStream_t stream) {
  ConvParams p = p_in;
  p.prof = g_prof_buf;
  p.debug_mode = g_debug_mode;
  const ConvEpilogue& e = p.e;
  const int f = feature_mask(e);
  // cout <= 64 layers run the M = 64 variant (conv_plan chose the ring geometry accordingly)
  const bool m64 = p.s.cout_pad <= 64;
  // ... and, with 3 x 3 taps over stationary weights, the variant whose MMA warp issues a tile's MMAs straight-line
  const bool stat = m64 && p.w_stationary && p.s.kw == 3 && p.s.kh == 3;
#define MVLM_CASE_BOTH(FLAGS) \
  case (FLAGS):               \
    return m64 ? (stat ? launch_t<(FLAGS) | F_M64 | F_STAT>(p, stream) : launch_t<(FLAGS) | F_M64>(p, stream)) : launch_t<(FLAGS)>(p, stream)
#define MVLM_CASE_128(FLAGS) \
  case (FLAGS):              \
    if (!m64) return launch_t<(FLAGS)>(p, stream); \
    break
  // the conv11 phase kernels: 2 x 2 taps over stationary weights at M = 128, straight-line issue as well
  if (f == F_ARGMAX && !m64 && p.w_stationary && p.s.kw == 2 && p.s.kh == 2) return launch_t<F_ARGMAX | F_STAT>(p, stream);
  switch (f) {
    // the combinations the network plan uses (hourglass.cu)
    MVLM_CASE_BOTH(F_PRE | F_RES1 | F_RAW | F_POST);  // RB conv1/2
    MVLM_CASE_BOTH(F_PRE | F_RES1 | F_RAW);
    MVLM_CASE_BOTH(F_RES1 | F_RAW | F_POST);          // RB conv3
    MVLM_CASE_BOTH(F_RES1 | F_RAW);
    MVLM_CASE_BOTH(F_RAW);                            // resample, conv6/10
    MVLM_CASE_128(F_PRE);                             // conv5, conv9
    MVLM_CASE_128(F_RES1 | F_RES2 | F_RAW | F_POST);  // conv7
    MVLM_CASE_128(F_ARGMAX);                          // conv11 phases
    MVLM_CASE_BOTH(F_F32);
    MVLM_CASE_BOTH(F_F32 | F_ARGMAX);
    MVLM_CASE_BOTH(F_MID | F_PRE | F_POST);           // stem (conv1)
    MVLM_CASE_BOTH(F_POOL | F_PRE | F_RES1 | F_RAW | F_POST);  // conv2 block: pooled outputs only
    MVLM_CASE_BOTH(F_POOL | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_POOL | F_RAW);
    MVLM_CASE_128(F_PRE | F_RES1 | F_RES2 | F_RAW | F_POST);
    // skip-branch ResidualBlocks with the up-sampled low path added in the epilogue (hourglass up path)
    MVLM_CASE_BOTH(F_UP | F_PRE | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_UP | F_PRE | F_RES1 | F_RAW);
    MVLM_CASE_BOTH(F_UP | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_UP | F_RES1 | F_RAW);
    // producers that also write the copies of a fused BatchNorm+ReLU / max-pool pass (aux_mode 1 / 2)
    MVLM_CASE_BOTH(F_POST2 | F_PRE | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_POST2 | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_POOLX | F_PRE | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_BOTH(F_POOLX | F_RES1 | F_RAW | F_POST);
    MVLM_CASE_128(F_POOLX | F_RES1 | F_RES2 | F_RAW | F_POST);
  }
#undef MVLM_CASE_BOTH
#undef MVLM_CASE_128
  set_error("conv_launch: unsupported epilogue combination 0x%x (cout_pad %d)", f, p.s.cout_pad);
  return MVLM_E_UNSUPPORTED;
}

}  // namespace mvlm
