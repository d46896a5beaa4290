// conv_wgrad_tc.cu -- convolution / linear weight gradients on the 5th-generation tensor cores.
//
//   dW^T[(tap, ci)][co]  =  sum over output pixels p of  x[p * stride + tap - pad][ci] * dy[p][co]
//
// is a GEMM whose reduction dimension is the PIXEL axis.  With NHWC activations both operands arrive with the
// reduction index as the row and the channel as the contiguous 128-byte swizzle row -- exactly what the forward's
// TMA boxes produce -- so the same shared-memory tiles are consumed as MN-major UMMA operands (instruction
// descriptor a_major = b_major = 1; canonical layout ((8,8,m),(8,k)):((1,8,LBO),(64,SBO)) in bf16 elements):
//   A (M = 128) = two (tap, 64-channel chunk) boxes of x, 16 KB apart (LBO);  rows = 128 pixels
//   B (N = BN)  = BN/64 boxes of dy, 16 KB apart;  in split-bf16 mode the lo plane follows the hi plane so one
//                 N = 2 BN instruction yields x_hi*dy_hi | x_hi*dy_lo and a second adds x_lo*dy_hi.
// One instruction consumes 16 pixels (two 8-row swizzle atoms, SBO = 1024 B): 8 instructions per 128-pixel tile.
// The pixel axis is split over gridDim.z; every CTA keeps its [128 x BN] fp32 accumulator in TMEM across its whole
// pixel range and writes one partial [co][K] slab; sbgm_wgrad_reduce sums the slabs in a fixed order
// (deterministic) into torch's OIHW layout.
// Warp roles as in conv_tc.cu: 0 = TMA producer, 1 = TMEM alloc + MMA issue, 2..5 = epilogue.
#include "tc_common.cuh"

namespace sbgm {

struct WgradParams {
  int n, ho, wo;
  int kh, kw, stride, pad;
  int w_tile, h_tile, n_tile, tiles_w, tiles_h, total_tiles;
  int cin_blocks, units, tiles_per_split, cout;
  size_t K;
  float* ws;     // [splits][cout][K]
};

constexpr uint32_t kBoxBytes = 128 * 128;   // 128 pixels x 64 bf16

template <int kSplit, int BN, int kStages>
struct WgradCfg {
  static constexpr uint32_t kABytes = kSplit * 2 * kBoxBytes;
  static constexpr uint32_t kBBytes = kSplit * (BN / 64) * kBoxBytes;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kBarOffset = kStages * kStageBytes;
  static constexpr uint32_t kSmemBytes = kBarOffset + 256 + 1024;
};

// MN-major operands: descriptor low word carries LBO = 16 KB (distance between 64-channel blocks)
__device__ __forceinline__ uint32_t desc_lo_mn(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | ((kBoxBytes >> 4) << 16); }
__device__ __forceinline__ constexpr uint32_t make_idesc_mn(int n) { return make_idesc(n) | (1u << 15) | (1u << 16); }

template <int FMT, int BN, int kStages>
__global__ void __launch_bounds__(192, 1)
conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy, const WgradParams p) {
  pdl_grid_sync();
  constexpr int kSplit = (FMT == SBGM_FMT_BF16X2) ? 2 : 1;
  using Cfg = WgradCfg<kSplit, BN, kStages>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + Cfg::kBarOffset;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * kStages);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 1);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_dy);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, kSplit * BN);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int u0 = blockIdx.x * 2;
  const bool second = (u0 + 1) < p.units;
  const int u1 = second ? u0 + 1 : u0;
  const int co0 = blockIdx.y * BN;
  const int tile_begin = blockIdx.z * p.tiles_per_split;
  const int tile_end = min(p.total_tiles, tile_begin + p.tiles_per_split);

  if (warp == 0) {
    if (lane == 0) {
      const int us[2] = {u0, u1};
      int r_[2], s_[2], cb_[2];
      for (int i = 0; i < 2; ++i) {
        const int tap = us[i] / p.cin_blocks;
        cb_[i] = us[i] - tap * p.cin_blocks;
        r_[i] = tap / p.kw;
        s_[i] = tap - r_[i] * p.kw;
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, tn = tile / (p.tiles_w * p.tiles_h);
        const int wo0 = tw * p.w_tile, ho0 = th * p.h_tile, n0 = tn * p.n_tile;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
        const uint32_t a_dst = smem_base + stage * Cfg::kStageBytes;
        const uint32_t b_dst = a_dst + Cfg::kABytes;
#pragma unroll
        for (int pl = 0; pl < kSplit; ++pl) {
#pragma unroll
          for (int i = 0; i < 2; ++i)
            tma_load_5d(a_dst + (pl * 2 + i) * kBoxBytes, &tmap_x, full_bar(stage), cb_[i] * 64, wo0 * p.stride + s_[i] - p.pad,
                        ho0 * p.stride + r_[i] - p.pad, n0, pl);
#pragma unroll
          for (int ch = 0; ch < BN / 64; ++ch)
            tma_load_5d(b_dst + (pl * (BN / 64) + ch) * kBoxBytes, &tmap_dy, full_bar(stage), co0 + ch * 64, wo0, ho0, n0, pl);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {     // one lane runs the issue loop (see conv_tc.cu)
      constexpr uint32_t idesc = make_idesc_mn(BN), idesc2 = make_idesc_mn(kSplit * BN);
      const uint64_t base = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo_mn(smem_base);
      uint32_t stage = 0, phase = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        mbar_wait(full_bar(stage), phase);
        tcgen05_fence_after();
        const uint64_t a0 = base + stage * (Cfg::kStageBytes >> 4);
        const uint64_t b0 = a0 + (Cfg::kABytes >> 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) {        // 8 x 16 pixels; 16 rows x 128 B = 2048 B per step
          if (kSplit == 2) {
            if (j == 0) umma_bf16(tmem_base, a0, b0, idesc2, tile != tile_begin);
            else umma_bf16_acc(tmem_base, a0 + j * 128, b0 + j * 128, idesc2);
            umma_bf16_acc(tmem_base, a0 + ((2 * kBoxBytes) >> 4) + j * 128, b0 + j * 128, idesc);
          } else {
            if (j == 0) umma_bf16(tmem_base, a0, b0, idesc, tile != tile_begin);
            else umma_bf16_acc(tmem_base, a0 + j * 128, b0 + j * 128, idesc);
          }
        }
        umma_commit(empty_bar(stage));
        if (tile == tile_end - 1) umma_commit(tmem_full_bar);
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int unit = (row < 64) ? u0 : u1;
    const bool valid = (row < 64) || second;
    const size_t kcol = static_cast<size_t>(unit) * 64 + (row & 63);
    float* dst = p.ws + (static_cast<size_t>(blockIdx.z) * p.cout + co0) * p.K + kcol;
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + c0;
      uint32_t r[32];
      tmem_ld32(taddr, r);
      if (kSplit == 2) {
        uint32_t t[32];
        tmem_ld32(taddr + BN, t);
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(__uint_as_float(r[j]) + __uint_as_float(t[j]));
      }
      if (valid) {
#pragma unroll
        for (int j = 0; j < 32; ++j) dst[static_cast<size_t>(c0 + j) * p.K] = __uint_as_float(r[j]);   // lanes <-> consecutive k: coalesced
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kSplit * BN);
}

// ---- 3x3 / stride 1 / pad 1 layers (bf16): halo-slab form ---------------------------------------------------------------
// The nine taps of one 64-channel block read the SAME activation pixels shifted by at most two rows / columns.  The kernel above
// fetches a 16 KB box per (tap, channel block) unit -- 144 KB of x per 128-pixel tile for the nine taps, by five CTAs -- and is
// bound by TMA latency times the bytes it can keep in flight (profiles/r02_ncu_wgrad_kernels_bf16.txt: tensor pipe 17-31 %, L2 and
// HBM far from saturated).  Here ONE CTA owns all nine taps of a channel block: per 16 x 8-pixel tile it loads one 18 x 10-pixel
// halo slab (23 KB, 128-byte-swizzle pixel rows as TMA writes them) and one dy box (16 KB), and every tap is a descriptor START
// inside the slab (conv3x3_c64.cu, conv_tc.cu slab mode) -- here for MN-major operands:
//   A (M = 128) = TWO taps of the channel block: start = slab + tap offset, LBO = the byte distance between the two taps' pixels
//                 (128 B, or 1024 B for the pair that wraps to the next slab row), SBO = the slab row pitch (10 pixels = 1280 B)
//                 between the 8-pixel atoms (= output rows); a 16-pixel K step is two output rows = 2560 B
//   B (N = 64)  = the dy box [128 pixels][64 channels], as before.
// Five accumulators [128 x 64] (tap pairs (0,1) (2,3) (4,5) (6,7) (8,8): the last pair computes tap 8 twice, its second half is
// not stored) live in 320 TMEM columns across the CTA's whole pixel range.  39 KB staged per 9.4 MFLOP instead of 240 KB.
constexpr uint32_t kWsSlabBytes = 25600;             // 18 x 10 pixels x 128 B = 23040, padded to a multiple of 1024
constexpr uint32_t kWsStageBytes = kWsSlabBytes + kBoxBytes;
constexpr int kWsStages = 5;
constexpr uint32_t kWsBarOffset = kWsStages * kWsStageBytes;
constexpr uint32_t kWsSmemBytes = kWsBarOffset + 256 + 1024;
constexpr uint32_t kWsSlabRow = 10 * 128;            // slab row pitch in bytes

struct WgradSlabParams {
  int tiles_w, tiles_h, total_tiles, tiles_per_split;
  int cin_blocks, cout;
  size_t K;
  float* ws;     // [splits][cout][K]
};

__global__ void __launch_bounds__(192, 1)
conv_wgrad_slab_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_dy, const WgradSlabParams p) {
  pdl_grid_sync();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + kWsBarOffset;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kWsStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * kWsStages);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kWsStages + 1);
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmap_x);
    tma_prefetch_desc(&tmap_dy);
    for (int s = 0; s < kWsStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  const int cb = blockIdx.x, co0 = blockIdx.y * 64;
  const int tile_begin = blockIdx.z * p.tiles_per_split;
  const int tile_end = min(p.total_tiles, tile_begin + p.tiles_per_split);

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        const int tw = tile % p.tiles_w, th = (tile / p.tiles_w) % p.tiles_h, n0 = tile / (p.tiles_w * p.tiles_h);
        const int wo0 = tw * 8, ho0 = th * 16;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_expect_tx(full_bar(stage), 18 * 10 * 128 + kBoxBytes);
        const uint32_t a_dst = smem_base + stage * kWsStageBytes;
        tma_load_5d(a_dst, &tmap_x, full_bar(stage), cb * 64, wo0 - 1, ho0 - 1, n0, 0);           // halo: out-of-bounds pixels zero-filled
        tma_load_5d(a_dst + kWsSlabBytes, &tmap_dy, full_bar(stage), co0, wo0, ho0, n0, 0);
        if (++stage == kWsStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_mn(64);
      // high descriptor words: SBO = slab row pitch for A, 1024 B for B; version 1, SWIZZLE_128B
      constexpr uint32_t kHiA = (kWsSlabRow >> 4) | (1u << 14) | (2u << 29);
      uint32_t stage = 0, phase = 0;
      for (int tile = tile_begin; tile < tile_end; ++tile) {
        mbar_wait(full_bar(stage), phase);
        tcgen05_fence_after();
        const uint32_t slab = smem_base + stage * kWsStageBytes;
        const uint64_t b0 = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo_mn(slab + kWsSlabBytes);
#pragma unroll
        for (int pr = 0; pr < 5; ++pr) {
          const int ta = 2 * pr, tb = pr == 4 ? 8 : 2 * pr + 1;
          const uint32_t off_a = ((ta / 3) * 10 + ta % 3) * 128, off_b = ((tb / 3) * 10 + tb % 3) * 128;
          const uint64_t a0 = (static_cast<uint64_t>(kHiA) << 32) | (((slab + off_a) & 0x3FFFFu) >> 4) | (((off_b - off_a) >> 4) << 16);
#pragma unroll
          for (int j = 0; j < 8; ++j) {        // 8 x 16 pixels: two output rows per step
            if (j == 0) umma_bf16(tmem_base + pr * 64, a0, b0, idesc, tile != tile_begin);
            else umma_bf16_acc(tmem_base + pr * 64, a0 + j * ((2 * kWsSlabRow) >> 4), b0 + j * 128, idesc);
          }
        }
        umma_commit(empty_bar(stage));
        if (tile == tile_end - 1) umma_commit(tmem_full_bar);
        if (++stage == kWsStages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int pr = 0; pr < 5; ++pr) {
      const int tap = 2 * pr + (row >> 6);
      const bool valid = tap < 9;
      const size_t kcol = (static_cast<size_t>(valid ? tap : 8) * p.cin_blocks + cb) * 64 + (row & 63);
      float* dst = p.ws + (static_cast<size_t>(blockIdx.z) * p.cout + co0) * p.K + kcol;
#pragma unroll 1
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + pr * 64 + c0, r);
        if (valid) {
#pragma unroll
          for (int j = 0; j < 32; ++j) dst[static_cast<size_t>(c0 + j) * p.K] = __uint_as_float(r[j]);
        }
      }
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

static void wgrad_slab_plan(int n, int h, int w, int cin, int cout, WgradSlabParams* p, int* splits) {
  p->tiles_w = w / 8; p->tiles_h = h / 16;
  p->total_tiles = n * p->tiles_w * p->tiles_h;
  p->cin_blocks = cin / 64; p->cout = cout;
  p->K = static_cast<size_t>(9) * cin;
  const int base = p->cin_blocks * (cout / 64);
  int s = (148 + base - 1) / base;                 // one wave of CTAs: every CTA dumps 5 x [128 x 64] fp32 = 160 KB of partials
  if (s > p->total_tiles) s = p->total_tiles;
  if (s < 1) s = 1;
  p->tiles_per_split = (p->total_tiles + s - 1) / s;
  *splits = (p->total_tiles + p->tiles_per_split - 1) / p->tiles_per_split;
}
// The slab form pays where a CTA's pixel range is long enough to amortise its 160 KB of partial sums (>= 8 tiles): measured on the
// C4 step, final conv_up 130 -> 89 us (870 TFLOP/s), the 64 x 64 layers 40 -> 33 us; the 32 x 32 and smaller 64 / 128-channel
// layers (2-4 tiles per CTA at one or two waves) came out equal or slower and stay on the per-unit kernel.
static bool wgrad_slab_ok(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad) {
  if (fmt != SBGM_FMT_BF16 || kh != 3 || kw != 3 || stride != 1 || pad != 1 || w % 8 != 0 || h % 16 != 0 || cin % 64 != 0 ||
      cout % 64 != 0)
    return false;
  WgradSlabParams sp;
  int ss = 0;
  wgrad_slab_plan(n, h, w, cin, cout, &sp, &ss);
  return sp.tiles_per_split >= 8;
}

static void wgrad_tc_plan(int n, int ho, int wo, int cin, int cout, int kh, int kw, int fmt, WgradParams* p, int* bn, int* splits) {
  p->n = n; p->ho = ho; p->wo = wo; p->kh = kh; p->kw = kw;
  pick_tile(n, ho, wo, &p->w_tile, &p->h_tile, &p->n_tile);
  p->tiles_w = ceil_div(wo, p->w_tile);
  p->tiles_h = ceil_div(ho, p->h_tile);
  p->total_tiles = p->tiles_w * p->tiles_h * ceil_div(n, p->n_tile);
  p->cin_blocks = cin / 64;
  p->units = kh * kw * p->cin_blocks;
  p->cout = cout;
  p->K = static_cast<size_t>(kh) * kw * cin;
  *bn = (fmt == SBGM_FMT_BF16 && cout % 128 == 0) ? 128 : 64;
  const int base = ((p->units + 1) / 2) * (cout / *bn);
  // pixel split: `waves` x 148 CTAs per layer.  Every CTA dumps its [128 x BN] fp32 accumulator and the reduce reads it back, so
  // the workspace traffic grows with the wave count.  Measured per layer on the C4 step (profiles/r02_wgrad_waves_*.txt): the
  // 64-wide layers (few CTAs per pixel range, long pixel ranges) are faster with three waves (final conv_up 130 vs 205 us), the
  // 128-wide ones (many (tap, channel-block) units) with one (36 launches: 362 vs 462 us, and a third of the reduce traffic).
  const int waves = *bn == 64 ? 3 : 1;
  int s = (148 * waves + base - 1) / base;
  if (s > p->total_tiles) s = p->total_tiles;
  if (s < 1) s = 1;
  p->tiles_per_split = (p->total_tiles + s - 1) / s;
  *splits = (p->total_tiles + p->tiles_per_split - 1) / p->tiles_per_split;
}

template <int FMT, int BN, int kStages>
static int launch_wgrad_tc(const CUtensorMap& tx, const CUtensorMap& td, const WgradParams& p, int splits, cudaStream_t st) {
  constexpr int kSplit = (FMT == SBGM_FMT_BF16X2) ? 2 : 1;
  using Cfg = WgradCfg<kSplit, BN, kStages>;
  auto kern = conv_wgrad_tc_kernel<FMT, BN, kStages>;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes) != cudaSuccess) {
      set_error("conv2d_wgrad_tc: cannot reserve %u bytes of shared memory", Cfg::kSmemBytes);
      return 1;
    }
    configured = true;
  }
  launch_k((kern), dim3((p.units + 1) / 2, p.cout / BN, splits), 192, Cfg::kSmemBytes, st, tx, td, p);
  return check_launch("conv2d_wgrad_tc");
}

}  // namespace sbgm

using namespace sbgm;

extern "C" size_t sbgm_conv2d_wgrad_tc_workspace_floats(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride,
                                                        int pad) {
  if (cin % 64 != 0 || cout % 64 != 0 || stride < 1) return 0;
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  if (ho <= 0 || wo <= 0) return 0;
  if (wgrad_slab_ok(fmt, n, h, w, cin, cout, kh, kw, stride, pad)) {
    WgradSlabParams sp;
    int ss = 0;
    wgrad_slab_plan(n, h, w, cin, cout, &sp, &ss);
    return static_cast<size_t>(ss) * cout * sp.K;
  }
  WgradParams p;
  int bn = 0, splits = 0;
  wgrad_tc_plan(n, ho, wo, cin, cout, kh, kw, fmt, &p, &bn, &splits);
  return static_cast<size_t>(splits) * cout * p.K;
}

extern "C" int sbgm_conv2d_wgrad_tc_plan(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, int* plan) {
  SBGM_REQUIRE(fmt == SBGM_FMT_BF16 || fmt == SBGM_FMT_BF16X2, "conv2d_wgrad_tc_plan: format %d is not a tensor-core format", fmt);
  SBGM_REQUIRE(cin % 64 == 0 && cout % 64 == 0, "conv2d_wgrad_tc_plan: cin=%d and cout=%d must be multiples of 64", cin, cout);
  SBGM_REQUIRE(stride >= 1 && stride <= 8, "conv2d_wgrad_tc_plan: stride %d unsupported", stride);
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  SBGM_REQUIRE(ho > 0 && wo > 0, "conv2d_wgrad_tc_plan: empty output");
  if (wgrad_slab_ok(fmt, n, h, w, cin, cout, kh, kw, stride, pad)) {
    WgradSlabParams sp;
    int ss = 0;
    wgrad_slab_plan(n, h, w, cin, cout, &sp, &ss);
    const int out[8] = {1, 64, ss, sp.tiles_per_split, sp.total_tiles, 8, 16, 1};
    for (int i = 0; i < 8; ++i) plan[i] = out[i];
    return 0;
  }
  WgradParams p;
  int bn = 0, splits = 0;
  wgrad_tc_plan(n, ho, wo, cin, cout, kh, kw, fmt, &p, &bn, &splits);
  SBGM_REQUIRE(p.w_tile * stride <= 256 && p.h_tile * stride <= 256, "conv2d_wgrad_tc_plan: TMA box too large for stride %d", stride);
  const int out[8] = {0, bn, splits, p.tiles_per_split, p.total_tiles, p.w_tile, p.h_tile, p.n_tile};
  for (int i = 0; i < 8; ++i) plan[i] = out[i];
  return 0;
}

extern "C" int sbgm_conv2d_wgrad_tc(const void* x, size_t x_plane, const void* dy, size_t dy_plane, float* dweight_oihw, int fmt,
                                    int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, float* workspace,
                                    void* stream) {
  SBGM_REQUIRE(fmt == SBGM_FMT_BF16 || fmt == SBGM_FMT_BF16X2, "conv2d_wgrad_tc: format %d is not a tensor-core format", fmt);
  SBGM_REQUIRE(cin % 64 == 0 && cout % 64 == 0, "conv2d_wgrad_tc: cin=%d and cout=%d must be multiples of 64", cin, cout);
  SBGM_REQUIRE(stride >= 1 && stride <= 8, "conv2d_wgrad_tc: stride %d unsupported", stride);
  SBGM_REQUIRE(dweight_oihw != nullptr, "conv2d_wgrad_tc: dweight_oihw is required");
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  SBGM_REQUIRE(ho > 0 && wo > 0, "conv2d_wgrad_tc: empty output");
  const int planes = (fmt == SBGM_FMT_BF16X2) ? 2 : 1;
  if (wgrad_slab_ok(fmt, n, h, w, cin, cout, kh, kw, stride, pad)) {
    WgradSlabParams sp;
    int ss = 0;
    wgrad_slab_plan(n, h, w, cin, cout, &sp, &ss);
    sp.ws = workspace;
    CUtensorMap sx, sd;
    if (encode_act_map(&sx, x, 1, x_plane, n, h, w, cin, 10, 18, 1, 1)) return 1;       // the 18 x 10-pixel halo slab
    if (encode_act_map(&sd, dy, 1, dy_plane, n, h, w, cout, 8, 16, 1, 1)) return 1;
    static bool configured = false;
    if (!configured) {
      if (cudaFuncSetAttribute(conv_wgrad_slab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWsSmemBytes) != cudaSuccess) {
        set_error("conv2d_wgrad_tc: cannot reserve %u bytes of shared memory", kWsSmemBytes);
        return 1;
      }
      configured = true;
    }
    launch_k((conv_wgrad_slab_kernel), dim3(sp.cin_blocks, cout / 64, ss), 192, kWsSmemBytes, as_stream(stream), sx, sd, sp);
    if (check_launch("conv2d_wgrad_tc")) return 1;
    return sbgm_wgrad_reduce(workspace, ss, cout, 9, cin, dweight_oihw, stream);
  }
  WgradParams p;
  int bn = 0, splits = 0;
  wgrad_tc_plan(n, ho, wo, cin, cout, kh, kw, fmt, &p, &bn, &splits);
  p.stride = stride; p.pad = pad; p.ws = workspace;
  SBGM_REQUIRE(p.w_tile * stride <= 256 && p.h_tile * stride <= 256, "conv2d_wgrad_tc: TMA box too large for stride %d", stride);
  CUtensorMap tx, td;
  if (encode_act_map(&tx, x, planes, x_plane, n, h, w, cin, p.w_tile, p.h_tile, p.n_tile, stride)) return 1;
  if (encode_act_map(&td, dy, planes, dy_plane, n, ho, wo, cout, p.w_tile, p.h_tile, p.n_tile, 1)) return 1;
  cudaStream_t st = as_stream(stream);
  int rc;
  if (fmt == SBGM_FMT_BF16) rc = (bn == 128) ? launch_wgrad_tc<SBGM_FMT_BF16, 128, 3>(tx, td, p, splits, st)
                                             : launch_wgrad_tc<SBGM_FMT_BF16, 64, 4>(tx, td, p, splits, st);
  else rc = launch_wgrad_tc<SBGM_FMT_BF16X2, 64, 2>(tx, td, p, splits, st);
  if (rc) return rc;
  return sbgm_wgrad_reduce(workspace, splits, cout, kh * kw, cin, dweight_oihw, stream);
}
