// conv_tc.cu -- convolution / linear layers as implicit GEMM on the 5th-generation tensor cores.
//
//   D[128 pixels x BLOCK_N channels] (fp32, TMEM)  +=  A[128 x 64] (smem, bf16)  *  B[BLOCK_N x 64]^T (smem, bf16)
//
// * A tiles are fetched straight from the NHWC activation tensor with one 5-D TMA box per filter
//   tap: box = (64 channels, w_tile, h_tile, n_tile, 1 plane) placed at
//   (cb*64, wo0*stride + s - pad, ho0*stride + r - pad, n0, plane).  Out-of-bounds pixels are
//   zero-filled by the TMA unit, which *is* the convolution's zero padding, and strided convolutions
//   use the tensor map's element strides -- no im2col buffer, no index arithmetic on the SMs.
//   The box lands in shared memory as 128 rows x 128 B with the 128-byte swizzle, exactly the
//   K-major canonical layout tcgen05.mma consumes.
// * B tiles come from the pre-packed weight matrix [planes][cout][kh*kw*cin] (K-major).
// * One elected thread issues tcgen05.mma (M=128, N=BLOCK_N, K=16) into a TMEM accumulator; a
//   kStages-deep mbarrier ring decouples TMA from MMA; four epilogue warps drain TMEM with
//   tcgen05.ld and apply bias / residual / activation / time-projection before the NHWC store.
// * BF16X2 ("split") activations and weights carry hi|lo bf16 planes; the three products
//   hi*hi + lo*hi + hi*lo accumulate into the same TMEM tile (fp32-class accuracy, 16-bit operands).
//
// Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = epilogue (warp w may only touch
// TMEM lanes 32*(w%4) .. +31).  Tiles with BLOCK_N >= 128 get a second epilogue group (warps 6..9, 320 threads) that
// takes the upper half of the columns: ncu showed a tile's epilogue (thousands of dependent instructions on one warp
// per scheduler) as long as the whole K loop of the mid-size layers, with nothing to overlap it at one CTA per SM.
#include "tc_common.cuh"

namespace sbgm {

struct ConvTcParams {
  int n, ho, wo;
  int kh, kw, stride, pad_h, pad_w;
  int out_h, out_w, out_step, out_oy, out_ox;   // scatter addressing of the output tensor (dgrad of strided convs)
  int w_tile, h_tile, n_tile;
  int tiles_w, tiles_h;
  int cin_blocks;
  int slab_perm;       // slab mode on 8 x 8 x 2-image tiles: tile rows ordered [h][n][w], tensor maps with (c, w, n, h) dims
  int slab_row;        // slab mode: descriptor units (16 B) per slab row step = pixels per slab row * 8
  uint32_t slab_tx;    // slab mode: bytes per slab plane
  int mt;              // pixel tiles per CTA (1 or 2; 2 = the MT = 2 kernels: two tiles share every weight box)
  int cluster;         // CTAs per cluster (1 or 2; 2 = slab mode with the weight boxes multicast over a CTA pair)
  int splits;          // split-K factor (gridDim.z); > 1 => raw fp32 partial tiles go to `ws`
  float* ws;           // [splits][pixels][cout] fp32
  float* gn_partials;  // [n][gn_chunks][cout/8][2] or nullptr: fused GroupNorm statistics (8-channel granularity)
  int gn_chunks;
  // LayerNorm folded into a Linear layer (LNF kernels): y = LN(x) W^T + b  ==  rstd_t (x W'^T - mean_t colsum) + b'  with
  // W' = W diag(gamma), b' = b + W beta, colsum_n = sum_c W'[n][c]; mean_t / rstd_t come from the A tiles as they pass through
  const float* ln_colsum;
  float ln_eps;
  EpilogueParams ep;
};

// ---- kernel ---------------------------------------------------------------------------------
template <int kAPl, int kBPl, int BLOCK_N, int kStages>
struct ConvTcCfg {
  static constexpr uint32_t kABytes = 128 * 128;               // 128 rows x 64 16-bit elements
  static constexpr uint32_t kBBytes = BLOCK_N * 128;
  static constexpr uint32_t kStageBytes = kAPl * kABytes + kBPl * kBBytes;
  static constexpr uint32_t kBarOffset = kStages * kStageBytes;
  static constexpr uint32_t kSmemBytes = kBarOffset + 256 + 1024;  // barriers + alignment slack
};

// Slab mode (3x3, stride 1, pad 1, maps tileable by 16 rows x 8 columns): the activation operand of a 64-channel block
// arrives ONCE as an 18 x 10-pixel halo slab and the nine taps are descriptor starts inside it (see conv3x3_c64.cu);
// only the weight boxes stream per tap.  Operand ingest per k-block drops from 16 KB + B to 2.5 KB + B (per plane).
constexpr int kSlabTileW = 8, kSlabTileH = 16, kSlabW = kSlabTileW + 2, kSlabH = kSlabTileH + 2, kSlabAStages = 2;
constexpr uint32_t kSlabPlaneBytes = 25600;                    // plane pitch in smem (1024-aligned): 18 x 10 or 10 x 2 x 10 pixels
constexpr uint32_t kDescHiSlab128 = ((kSlabW * 128u) >> 4) | (1u << 14) | (2u << 29);   // SBO = one slab row
template <int kAPl, int kBPl, int BLOCK_N, int kStages>
struct ConvTcSlabCfg {
  static constexpr uint32_t kBBytes = BLOCK_N * 128;
  static constexpr uint32_t kAStageBytes = kAPl * kSlabPlaneBytes;
  static constexpr uint32_t kBStageBytes = kBPl * kBBytes;
  static constexpr uint32_t kBOffset = kSlabAStages * kAStageBytes;
  static constexpr uint32_t kBarOffset = kBOffset + kStages * kBStageBytes;
  static constexpr uint32_t kSmemBytes = kBarOffset + 256 + 1024;
};

template <int BLOCK_N>
struct ConvTcThreads {
  static constexpr int kEpiGroups = BLOCK_N >= 128 ? 2 : 1;
  static constexpr int kThreads = 64 + 128 * kEpiGroups;
  static constexpr int kMinCtas = BLOCK_N >= 128 ? 1 : 2;
};

// MT = pixel tiles per CTA (1 or 2).  With MT = 2 a CTA owns two consecutive 128-pixel tiles that share every weight box: the
// K-heavy layers are bound by the chip-wide L2 -> SM bandwidth (ncu: ~30 B/clk per SM with all SMs pulling, tensor pipe 25-48 %),
// and two thirds to nine tenths of their operand bytes are weights that every pixel tile re-fetches.
// CL = CTAs per cluster (1 or 2; slab mode only).  With CL = 2 the two CTAs of a cluster own different pixel tiles of the SAME
// output-channel block and K range, so they consume the same weight stream: each loads HALF of every weight box and multicasts it
// into both CTAs' stage (the L2 -> SM weight traffic, two thirds to nine tenths of a K-heavy layer's operand bytes, halves).
// A weight stage may be rewritten only when BOTH consumers have released it: the MMA issuer's commit arrives on the `empty`
// barrier of both CTAs (count 2).  The activation slabs and everything else stay per CTA.
template <int FMT, int BLOCK_N, int kStages, int ACT, int PROJ, bool STAGED, bool SLAB = false, bool LNF = false, int MT = 1, int CL = 1>
__global__ void __launch_bounds__(ConvTcThreads<BLOCK_N>::kThreads, ConvTcThreads<BLOCK_N>::kMinCtas)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_o, const ConvTcParams p) {
  pdl_grid_sync();
  // kAPl activation planes (2: split-bf16 hi|lo), kBPl weight planes (2: hi|lo, adjacent in a stage so that ONE MMA of width
  // 2 * BLOCK_N multiplies an activation plane with both; F16: w_lo is stored times 2^11 and the epilogue rescales its half)
  constexpr int kAPl = TcFmt<FMT>::kAPlanes, kBPl = TcFmt<FMT>::kBPlanes;
  using Cfg = ConvTcCfg<kAPl * MT, kBPl, BLOCK_N, kStages>;          // a stage holds the A tiles of all MT pixel tiles
  using SCfg = ConvTcSlabCfg<kAPl * MT, kBPl, BLOCK_N, kStages>;
  constexpr uint32_t kAccCols = kBPl * BLOCK_N;                       // accumulator columns of one pixel tile
  constexpr uint32_t kATile = kAPl * Cfg::kABytes, kSlabTile = kAPl * kSlabPlaneBytes;   // bytes of one pixel tile's A operand
  static_assert(MT * kAccCols <= 512, "accumulators exceed the 512 TMEM columns");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_base = smem_base + (SLAB ? SCfg::kBarOffset : Cfg::kBarOffset);
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
  const uint32_t tmem_full_bar = bar_base + 8u * (2 * kStages);
  const uint32_t tmem_slot = bar_base + 8u * (2 * kStages + 1);
  auto slab_full = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + s); };                   // slab mode only
  auto slab_empty = [&](int s) { return bar_base + 8u * (2 * kStages + 2 + kSlabAStages + s); };
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  static_assert(CL == 1 || (CL == 2 && SLAB && !LNF && !PROJ), "clusters: slab mode only");
  const uint32_t cta_rank = CL > 1 ? cluster_ctarank() : 0u;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar(s), 1);
      // LNF: the epilogue warps read every A tile too (row statistics) and release the stage together with the MMA
      // CL = 2: the stage is shared by the cluster's two consumers
      mbar_init(empty_bar(s), LNF ? 1 + 4 * ConvTcThreads<BLOCK_N>::kEpiGroups : CL);
    }
    mbar_init(tmem_full_bar, 1);
    if (SLAB) {
      for (int s = 0; s < kSlabAStages; ++s) {
        mbar_init(slab_full(s), 1);
        mbar_init(slab_empty(s), 1);
      }
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, MT * kAccCols);
  tcgen05_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();      // the peer's barriers exist before anything is multicast into this CTA or arrives on them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  // tile coordinates (pixel tiles blockIdx.x * MT + m; a tile past the last one lies outside the tensor: TMA zero-fills its
  // operand and clips its stores)
  int tw_[MT], th_[MT], wo0_[MT], ho0_[MT], n0_[MT];
#pragma unroll
  for (int m = 0; m < MT; ++m) {
    const int mt = blockIdx.x * MT + m;
    tw_[m] = mt % p.tiles_w;
    th_[m] = (mt / p.tiles_w) % p.tiles_h;
    wo0_[m] = tw_[m] * p.w_tile;
    ho0_[m] = th_[m] * p.h_tile;
    n0_[m] = (mt / (p.tiles_w * p.tiles_h)) * p.n_tile;
  }
  const int co0 = blockIdx.y * BLOCK_N;
  const int total_kb = p.kh * p.kw * p.cin_blocks;
  const int kb_per = (total_kb + p.splits - 1) / p.splits;
  const int kb_begin = blockIdx.z * kb_per;
  const int num_kb = min(total_kb, kb_begin + kb_per) - kb_begin;     // >= 1 by construction of `splits`
  // slab mode splits K by 64-channel blocks (each block = nine taps of one slab)
  const int cb_per = (p.cin_blocks + p.splits - 1) / p.splits;
  const int cb_begin = blockIdx.z * cb_per;
  const int cb_cnt = min(p.cin_blocks, cb_begin + cb_per) - cb_begin;  // >= 1: checked by the host

  if (SLAB && warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int i = 0; i < cb_cnt; ++i) {
        const int cb = cb_begin + i, as = i & 1;
        mbar_wait(slab_empty(as), ((i >> 1) & 1u) ^ 1u);
        mbar_expect_tx(slab_full(as), MT * kAPl * p.slab_tx);
#pragma unroll
        for (int m = 0; m < MT; ++m)
#pragma unroll
          for (int pl = 0; pl < kAPl; ++pl)
            tma_load_5d(smem_base + as * SCfg::kAStageBytes + m * kSlabTile + pl * kSlabPlaneBytes, &tmap_a, slab_full(as), cb * 64,
                        wo0_[m] - 1, p.slab_perm ? n0_[m] : ho0_[m] - 1, p.slab_perm ? ho0_[m] - 1 : n0_[m], pl);
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(empty_bar(stage), phase ^ 1u);
          mbar_expect_tx(full_bar(stage), SCfg::kBStageBytes);
          const uint32_t b_dst = smem_base + SCfg::kBOffset + stage * SCfg::kBStageBytes;
#pragma unroll
          for (int pl = 0; pl < kBPl; ++pl) {
            if (CL > 1)      // this CTA's half of the rows, into both CTAs' stage (tmap_b's box is BLOCK_N / 2 rows)
              tma_load_3d_multicast(b_dst + pl * SCfg::kBBytes + cta_rank * (BLOCK_N / 2) * 128u, &tmap_b, full_bar(stage),
                                    (tap * p.cin_blocks + cb) * 64, co0 + static_cast<int>(cta_rank) * (BLOCK_N / 2), pl, 0x3);
            else
              tma_load_3d(b_dst + pl * SCfg::kBBytes, &tmap_b, full_bar(stage), (tap * p.cin_blocks + cb) * 64, co0, pl);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (SLAB && warp == 1) {
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(BLOCK_N, TcFmt<FMT>::kHalf), idesc2 = make_idesc(kBPl * BLOCK_N, TcFmt<FMT>::kHalf);
      const uint64_t a_base = (static_cast<uint64_t>(kDescHiSlab128) << 32) | desc_lo(smem_base);
      const uint64_t b_base = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo(smem_base + SCfg::kBOffset);
      uint32_t stage = 0, phase = 0;
      for (int i = 0; i < cb_cnt; ++i) {
        const int as = i & 1;
        mbar_wait(slab_full(as), (i >> 1) & 1u);
        tcgen05_fence_after();
        const uint64_t a_slab = a_base + as * (SCfg::kAStageBytes >> 4);
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          mbar_wait(full_bar(stage), phase);
          tcgen05_fence_after();
          // tap (r, s): the 128 A rows start at slab pixel (r, s); 8-row groups (output rows) are one slab row apart
          const uint64_t a0 = a_slab + static_cast<uint32_t>((tap / 3) * p.slab_row + (tap % 3) * 8);
          const uint64_t b0 = b_base + stage * (SCfg::kBStageBytes >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int m = 0; m < MT; ++m) {
              const uint64_t am = a0 + m * (kSlabTile >> 4);
              const uint32_t dm = tmem_base + m * kAccCols;
              if (k == 0 && tap == 0) umma_bf16(dm, am, b0, idesc2, i != 0);
              else umma_bf16_acc(dm, am + 2 * k, b0 + 2 * k, idesc2);
              if (kAPl == 2) umma_bf16_acc(dm, am + (kSlabPlaneBytes >> 4) + 2 * k, b0 + 2 * k, idesc);
            }
          }
          if (CL > 1) umma_commit_multicast(empty_bar(stage), 0x3); else umma_commit(empty_bar(stage));
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
        umma_commit(slab_empty(as));
      }
      umma_commit(tmem_full_bar);
    }
    __syncwarp();
  } else if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kbi = 0; kbi < num_kb; ++kbi) {
        const int kb = kb_begin + kbi;
        const int tap = kb / p.cin_blocks, cb = kb - tap * p.cin_blocks;
        const int r = tap / p.kw, s = tap - r * p.kw;
        mbar_wait(empty_bar(stage), phase ^ 1u);
        mbar_expect_tx(full_bar(stage), Cfg::kStageBytes);
        const uint32_t a_dst = smem_base + stage * Cfg::kStageBytes;
        const uint32_t b_dst = a_dst + MT * kATile;
#pragma unroll
        for (int m = 0; m < MT; ++m)
#pragma unroll
          for (int pl = 0; pl < kAPl; ++pl)
            tma_load_5d(a_dst + m * kATile + pl * Cfg::kABytes, &tmap_a, full_bar(stage), cb * 64, wo0_[m] * p.stride + s - p.pad_w,
                        ho0_[m] * p.stride + r - p.pad_h, n0_[m], pl);
#pragma unroll
        for (int pl = 0; pl < kBPl; ++pl) tma_load_3d(b_dst + pl * Cfg::kBBytes, &tmap_b, full_bar(stage), kb * 64, co0, pl);
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // one elected lane runs the whole issue loop (64-bit descriptors, ~3 instructions per MMA; the earlier
    // warp-uniform variant paid an election, a predicate vote and four register->uniform moves per MMA)
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc(BLOCK_N, TcFmt<FMT>::kHalf), idesc2 = make_idesc(kBPl * BLOCK_N, TcFmt<FMT>::kHalf);
      const uint64_t base = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo(smem_base);
      uint32_t stage = 0, phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(full_bar(stage), phase);
        tcgen05_fence_after();
        const uint64_t a0 = base + stage * (Cfg::kStageBytes >> 4);
        const uint64_t b0 = a0 + ((MT * kATile) >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // 4 x (K = 16 elements = 32 B) per 64-element block
          // two weight planes (hi|lo) of a stage are adjacent: one N = 2*BLOCK_N MMA yields x*w_hi (first half of the
          // columns) and x*w_lo (second half); split-bf16 adds x_lo*w_hi into the first half.
#pragma unroll
          for (int m = 0; m < MT; ++m) {
            const uint64_t am = a0 + m * (kATile >> 4);
            const uint32_t dm = tmem_base + m * kAccCols;
            if (k == 0) umma_bf16(dm, am, b0, idesc2, kb != 0);
            else umma_bf16_acc(dm, am + 2 * k, b0 + 2 * k, idesc2);
            if (kAPl == 2) umma_bf16_acc(dm, am + (Cfg::kABytes >> 4) + 2 * k, b0 + 2 * k, idesc);
          }
        }
        umma_commit(empty_bar(stage));          // frees the smem slot once these MMAs retire
        if (kb == num_kb - 1) umma_commit(tmem_full_bar);
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
    }
    __syncwarp();
  } else {
    // ---- epilogue: TMEM -> registers -> bias/residual/act/time -> NHWC global ----
    const int quarter = warp & 3;
    constexpr int kColsPerGroup = BLOCK_N / ConvTcThreads<BLOCK_N>::kEpiGroups;
    const int c_begin = ((warp - 2) >> 2) * kColsPerGroup, c_end = c_begin + kColsPerGroup;
    const int row = quarter * 32 + lane;
    int w_l = row % p.w_tile, h_l = (row / p.w_tile) % p.h_tile, n_l = row / (p.w_tile * p.h_tile);
    if (SLAB && p.slab_perm) {          // tile rows ordered [h][n][w]
      n_l = (row / p.w_tile) % p.n_tile;
      h_l = row / (p.w_tile * p.n_tile);
    }
    float proj_acc[kProjMax];
#pragma unroll
    for (int q = 0; q < kProjMax; ++q) proj_acc[q] = 0.0f;
    float ln_mean = 0.0f, ln_rstd = 1.0f;
    if (LNF) {
      // LayerNorm statistics of this thread's row (token) over ALL input channels, read from the A tiles while the MMA consumes
      // them: 64 channels per k-block, 16-byte chunks at the 128-byte-swizzle positions TMA wrote them to
      // two channels per instruction (FADD2 / FFMA2): (even, odd) partial sums, added at the end
      unsigned long long sum2 = 0ull, sq2 = 0ull;
      uint32_t stage = 0, phase = 0;
      for (int kbi = 0; kbi < num_kb; ++kbi) {
        mbar_wait(full_bar(stage), phase);
        const uint32_t a_row = smem_base + stage * Cfg::kStageBytes + row * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
          for (int pl = 0; pl < kAPl; ++pl) {
            uint4 u;
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w)
                         : "r"(a_row + pl * Cfg::kABytes + ((j ^ (row & 7)) << 4)));
            float t[8];
            if (TcFmt<FMT>::kHalf) unpack_f16x8(u, t); else unpack_bf16x8(u, t);
#pragma unroll
            for (int e = 0; e < 8; ++e) v[e] += t[e];
          }
#pragma unroll
          for (int e = 0; e < 8; e += 2) {
            unsigned long long vp;
            asm("mov.b64 %0, {%1, %2};" : "=l"(vp) : "f"(v[e]), "f"(v[e + 1]));
            asm("add.rn.f32x2 %0, %0, %1;" : "+l"(sum2) : "l"(vp));
            asm("fma.rn.f32x2 %0, %1, %1, %0;" : "+l"(sq2) : "l"(vp));
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar(stage));
        if (++stage == kStages) { stage = 0; phase ^= 1u; }
      }
      float s0, s1, q0, q1;
      asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(sum2));
      asm("mov.b64 {%0, %1}, %2;" : "=f"(q0), "=f"(q1) : "l"(sq2));
      const float sum = s0 + s1, sq = q0 + q1;
      const float inv_c = 1.0f / static_cast<float>(p.cin_blocks * 64);
      ln_mean = sum * inv_c;
      ln_rstd = rsqrtf(fmaxf(sq * inv_c - ln_mean * ln_mean, 0.0f) + p.ln_eps);
    }
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
#pragma unroll 1
    for (int m = 0; m < MT; ++m) {
    const int tw = tw_[m], th = th_[m], wo0 = wo0_[m], ho0 = ho0_[m], n0 = n0_[m];
    const int n = n0 + n_l, oy = ho0 + h_l, ox = wo0 + w_l;
    const bool valid = (n < p.n) && (oy < p.ho) && (ox < p.wo);
    const size_t pix = (static_cast<size_t>(n) * p.out_h + oy * p.out_step + p.out_oy) * p.out_w + ox * p.out_step + p.out_ox;
    if (MT > 1 && m > 0 && STAGED) {      // the warp's staging area is re-used: the previous tile's bulk stores must have read it
      if (lane == 0) tma_store_wait_read();
      __syncwarp();
    }
    auto load_acc = [&](int c0, uint32_t (&r)[32]) {
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + m * kAccCols + c0;
      tmem_ld32(taddr, r);
      if (kBPl == 2) {
        uint32_t t[32];
        tmem_ld32(taddr + BLOCK_N, t);
        merge_lo<FMT>(r, t);
      }
    };
    if (!PROJ && p.splits > 1) {                    // split-K: raw fp32 partial tile, finished by splitk_finalize_kernel
      float* dst = p.ws + (static_cast<size_t>(blockIdx.z) * p.n * p.ho * p.wo + pix) * p.ep.cout + co0;
#pragma unroll 1
      for (int c0 = c_begin; c0 < c_end; c0 += 32) {
        uint32_t ra[32];
        load_acc(c0, ra);
        if (valid) {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            reinterpret_cast<float4*>(dst + c0)[j] = make_float4(__uint_as_float(ra[4 * j]), __uint_as_float(ra[4 * j + 1]),
                                                                 __uint_as_float(ra[4 * j + 2]), __uint_as_float(ra[4 * j + 3]));
        }
      }
    } else {
#pragma unroll 1
      for (int c0 = c_begin; c0 < c_end; c0 += 64) {  // the whole warp walks its share of the tile in 64-channel blocks
        uint32_t ra[32], rb[32];
        load_acc(c0, ra);
        load_acc(c0 + 32, rb);
        if (LNF) {
          // rstd * (acc - mean * colsum), four column sums per load, two columns per instruction
          const float4* cs = reinterpret_cast<const float4*>(p.ln_colsum + co0 + c0);
          unsigned long long nm2, rs2;
          asm("mov.b64 %0, {%1, %1};" : "=l"(nm2) : "f"(-ln_mean));
          asm("mov.b64 %0, {%1, %1};" : "=l"(rs2) : "f"(ln_rstd));
          auto fold = [&](uint32_t& x0, uint32_t& x1, float c0_, float c1_) {
            unsigned long long a, c;
            asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(x0), "r"(x1));
            asm("mov.b64 %0, {%1, %2};" : "=l"(c) : "f"(c0_), "f"(c1_));
            asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(nm2), "l"(c));
            asm("mul.rn.f32x2 %0, %0, %1;" : "+l"(a) : "l"(rs2));
            asm("mov.b64 {%0, %1}, %2;" : "=r"(x0), "=r"(x1) : "l"(a));
          };
#pragma unroll
          for (int g = 0; g < 8; ++g) {
            const float4 ca = __ldg(cs + g), cb = __ldg(cs + 8 + g);
            fold(ra[4 * g], ra[4 * g + 1], ca.x, ca.y);
            fold(ra[4 * g + 2], ra[4 * g + 3], ca.z, ca.w);
            fold(rb[4 * g], rb[4 * g + 1], cb.x, cb.y);
            fold(rb[4 * g + 2], rb[4 * g + 3], cb.z, cb.w);
          }
        }
        if (!PROJ && p.gn_partials) {
          // this warp's 32 rows lie in one image (host-checked): chunk = which 32-row strip of that image
          int img, chunk;
          if (p.n_tile == 1) {
            img = n0;
            chunk = (th * p.tiles_w + tw) * 4 + quarter;
          } else {
            const int rows_per_img = p.h_tile * p.w_tile;
            img = n0 + (quarter * 32) / rows_per_img;
            chunk = ((quarter * 32) % rows_per_img) >> 5;
          }
          if (img < p.n)
            gn_block64_stats<FMT>(ra, rb, p.ep.bias, co0 + c0, valid, lane,
                                  p.gn_partials + ((static_cast<size_t>(img) * p.gn_chunks + chunk) * (p.ep.cout >> 3) + ((co0 + c0) >> 3)) * 2);
        }
        StageArgs sa;
        if (STAGED) {
          // the pipeline stages are free once tmem_full has fired (every MMA, hence every operand read, has retired):
          // warp e stages its 64-column blocks (x planes) back to back from smem_base + e * kWarpStride
          const int r0 = quarter * 32;
          sa.tmap_o = &tmap_o;
          constexpr uint32_t kBlockStride = kAPl * kStageBlockBytes, kWarpStride = (kColsPerGroup / 64) * kBlockStride;
          sa.stage = smem_base + static_cast<uint32_t>(warp - 2) * kWarpStride + static_cast<uint32_t>((c0 - c_begin) >> 6) * kBlockStride;
          sa.x0 = wo0 + r0 % p.w_tile;
          sa.y0 = ho0 + (r0 / p.w_tile) % p.h_tile;
          sa.n0 = n0 + r0 / (p.w_tile * p.h_tile);
          if (SLAB && p.slab_perm) {    // output map dims (c, w, n, h): the warp's 32 rows are [2 h][2 n][8 w]
            sa.y0 = n0;
            sa.n0 = ho0 + r0 / (p.w_tile * p.n_tile);
          }
        }
        epilogue_block64<FMT, ACT, PROJ, STAGED>(p.ep, ra, rb, co0 + c0, n, pix, valid, lane, proj_acc, sa);
      }
    }
    if (PROJ && valid) epilogue_store_proj(p.ep, pix, proj_acc);
    }     // pixel tiles
    if (STAGED && !(!PROJ && p.splits > 1) && lane == 0) tma_store_wait_read();      // the staged tiles must be read out before the CTA retires
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();      // no CTA retires while its peer may still multicast into it or arrive on its barriers
  if (warp == 1) tmem_dealloc(tmem_base, MT * kAccCols);
}

// Sum the split-K partial tiles in a fixed order (deterministic) and apply the fused epilogue.
template <int FMT, int ACT>
__global__ void splitk_finalize_kernel(const float* __restrict__ ws, int splits, size_t pixels, int hw, EpilogueParams ep) {
  pdl_grid_sync();
  const int vecs = ep.cout >> 3;
  const size_t total = pixels * vecs;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const size_t pix = i / vecs;
    const int co = static_cast<int>(i % vecs) * 8;
    float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int z = 0; z < splits; ++z) {
      const float4* src = reinterpret_cast<const float4*>(ws + (static_cast<size_t>(z) * pixels + pix) * ep.cout + co);
      const float4 a = __ldg(src), b = __ldg(src + 1);
      v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w; v[4] += b.x; v[5] += b.y; v[6] += b.z; v[7] += b.w;
    }
    if (ep.bias) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += __ldg(ep.bias + co + j);
    }
    if (ep.residual) {
      float rv[8];
      Act<FMT>::load8(ep.residual, ep.res_plane, (ep.res_pix_mod ? pix % ep.res_pix_mod : pix) * ep.cout + co, rv);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += rv[j];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = act_ct<ACT>(v[j]);
    if (ep.tproj) {
      const int n = static_cast<int>(pix / hw);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += __ldg(ep.tproj + static_cast<size_t>(n) * ep.tproj_stride + co + j);
    }
    Act<FMT>::store8(ep.out, ep.out_plane, pix * ep.cout + co, v);
  }
}

// ---- host side ---------------------------------------------------------------------------------
EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(ptr);
  return fn;
}

int encode_act_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int n, int h, int w, int c,
                   int box_w, int box_h, int box_n, int stride, int box_c) {
  EncodeTiledFn encode = get_encode_fn();
  SBGM_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled unavailable (driver too old?)");
  const cuuint64_t dims[5] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n, (cuuint64_t)planes};
  const cuuint64_t strides[4] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2,
                                 planes == 2 ? (cuuint64_t)plane_elems * 2 : (cuuint64_t)n * h * w * c * 2};
  SBGM_REQUIRE(box_c == 64 || box_c == 32, "encode_act_map: box_c must be 64 or 32");
  const cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)(box_w * stride), (cuuint32_t)(box_h * stride), (cuuint32_t)box_n, 1};
  const cuuint32_t estr[5] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, box_c == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SBGM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(activations) failed with %d", (int)r);
  return 0;
}

int encode_out_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int n, int h, int w, int c,
                   int tile_w, int tile_h, int tile_n) {
  EncodeTiledFn encode = get_encode_fn();
  SBGM_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled unavailable (driver too old?)");
  // 32 consecutive tile rows (w fastest, then h, then n) form a rectangular sub-box because every tile extent is a power of two
  const int bw = tile_w >= 32 ? 32 : tile_w;
  const int bh = tile_w >= 32 ? 1 : (tile_w * tile_h >= 32 ? 32 / tile_w : tile_h);
  const int bn = 32 / (bw * bh);
  (void)tile_n;
  const cuuint64_t dims[5] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n, (cuuint64_t)planes};
  const cuuint64_t strides[4] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2,
                                 planes == 2 ? (cuuint64_t)plane_elems * 2 : (cuuint64_t)n * h * w * c * 2};
  const cuuint32_t box[5] = {64, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SBGM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(output) failed with %d", (int)r);
  return 0;
}

// NHWC tensor seen with dims (c, w, n, h, plane): a box (64, box_w, box_n, box_h) lands in shared memory ordered [h][n][w], so
// that row groups of a tile spanning several images stay one slab row apart (slab mode on 8 x 8 maps).  Used for the halo slab
// (box 10 x 2 x 10) and for the staged output store (box 8 x 2 x 2 = one warp's 32 rows).
static int encode_perm_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int n, int h, int w, int c,
                           int box_w, int box_n, int box_h) {
  EncodeTiledFn encode = get_encode_fn();
  SBGM_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled unavailable (driver too old?)");
  const cuuint64_t dims[5] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)n, (cuuint64_t)h, (cuuint64_t)planes};
  const cuuint64_t strides[4] = {(cuuint64_t)c * 2, (cuuint64_t)h * w * c * 2, (cuuint64_t)w * c * 2,
                                 planes == 2 ? (cuuint64_t)plane_elems * 2 : (cuuint64_t)n * h * w * c * 2};
  const cuuint32_t box[5] = {64, (cuuint32_t)box_w, (cuuint32_t)box_n, (cuuint32_t)box_h, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SBGM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(permuted) failed with %d", (int)r);
  return 0;
}

int encode_weight_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int cout, int K, int box_rows) {
  EncodeTiledFn encode = get_encode_fn();
  SBGM_REQUIRE(encode != nullptr, "cuTensorMapEncodeTiled unavailable (driver too old?)");
  const cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)cout, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)K * 2, planes == 2 ? (cuuint64_t)plane_elems * 2 : (cuuint64_t)K * cout * 2};
  const cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  SBGM_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(weights) failed with %d", (int)r);
  return 0;
}

static int pow2_floor(int v) { int p = 1; while (p * 2 <= v) p *= 2; return p; }
static int pow2_ceil(int v) { int p = 1; while (p < v) p *= 2; return p; }
static int pow2_divisor(int v) { return v & (-v); }

// Pick (w_tile, h_tile, n_tile), product 128, powers of two, covering the output with the least padding.
void pick_tile(int n, int ho, int wo, int* wt, int* ht, int* nt) {
  if (ho == 1 && n == 1) {  // token matrix [M][C] (Linear layers): plain 128-row tiles, tail masked
    *wt = 128; *ht = 1; *nt = 1;
    return;
  }
  int w_tile = pow2_divisor(wo);
  if (w_tile > 128) w_tile = 128;
  if (w_tile < 8 && wo > w_tile) w_tile = pow2_ceil(wo) > 128 ? 128 : pow2_ceil(wo);
  int rest = 128 / w_tile;
  int h_tile = pow2_divisor(ho);
  if (h_tile > rest) h_tile = rest;
  if (h_tile < rest && ho > h_tile && pow2_divisor(ho) < 4) h_tile = pow2_ceil(ho) > rest ? rest : pow2_ceil(ho);
  *wt = w_tile;
  *ht = h_tile;
  *nt = rest / h_tile;
  (void)n;
  (void)pow2_floor;
}

template <int FMT, int BLOCK_N, int kStages, int ACT, int PROJ, bool STAGED, bool SLAB = false, bool LNF = false, int MT = 1, int CL = 1>
static int launch_conv_tc_inst(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const ConvTcParams& p, int m_tiles,
                               cudaStream_t st) {
  constexpr int kAPl = TcFmt<FMT>::kAPlanes, kBPl = TcFmt<FMT>::kBPlanes;
  using Cfg = std::conditional_t<SLAB, ConvTcSlabCfg<kAPl * MT, kBPl, BLOCK_N, kStages>, ConvTcCfg<kAPl * MT, kBPl, BLOCK_N, kStages>>;
  static_assert(!STAGED || Cfg::kBarOffset >= 4u * (BLOCK_N / 64) * kAPl * kStageBlockBytes, "the staging area must fit in the pipeline stages");
  static_assert(MT * kBPl * BLOCK_N <= 512, "accumulator exceeds the 512 TMEM columns");
  static_assert(Cfg::kSmemBytes <= 232448, "shared memory budget");
  auto kern = conv_tc_kernel<FMT, BLOCK_N, kStages, ACT, PROJ, STAGED, SLAB, LNF, MT, CL>;
  static bool configured = false;
  if (!configured) {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes) != cudaSuccess) {
      set_error("conv2d_tc: cannot reserve %u bytes of shared memory", Cfg::kSmemBytes);
      return 1;
    }
    configured = true;
  }
  if (PROJ && cudaMemcpyToSymbolAsync(c_proj_w, p.ep.proj_w, sizeof(float) * kProjN * 64, 0, cudaMemcpyDeviceToDevice, st) != cudaSuccess) {
    set_error("conv2d_tc: projection weight upload failed");
    return 1;
  }
  dim3 grid((m_tiles + MT - 1) / MT, p.ep.cout / BLOCK_N, p.splits);
  if (CL > 1) {        // whole clusters: a CTA past the last pixel tile computes on zero-filled operands and stores nothing
    grid.x = (grid.x + CL - 1) / CL * CL;
    launch_k_cluster((kern), grid, ConvTcThreads<BLOCK_N>::kThreads, Cfg::kSmemBytes, st, CL, ta, tb, to, p);
  } else {
    launch_k((kern), grid, ConvTcThreads<BLOCK_N>::kThreads, Cfg::kSmemBytes, st, ta, tb, to, p);
  }
  if (!PROJ && p.splits > 1) {
    const size_t pixels = static_cast<size_t>(p.n) * p.ho * p.wo;
    const size_t items = pixels * (p.ep.cout / 8);
    const int fgrid = static_cast<int>(items / 256 + 1 < 148 * 8 ? items / 256 + 1 : 148 * 8);
    launch_k((splitk_finalize_kernel<FMT, ACT>), fgrid, 256, 0, st, p.ws, p.splits, pixels, p.ho * p.wo, p.ep);
  }
  return check_launch("conv2d_tc");
}

template <int FMT, int BLOCK_N, int kStages>
static int launch_conv_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const ConvTcParams& p, int m_tiles,
                          cudaStream_t st) {
  if (p.ln_colsum) {          // LayerNorm-folded Linear layers (in_proj: no activation; ff.0: GELU), staged store only
    if (BLOCK_N > 128 || !p.ep.staged) { set_error("conv2d_tc: the LayerNorm-folded form needs 64/128-wide staged tiles"); return 1; }
    constexpr int BN = BLOCK_N > 128 ? 128 : BLOCK_N;
    if (p.ep.act == SBGM_ACT_NONE) return launch_conv_tc_inst<FMT, BN, kStages, SBGM_ACT_NONE, 0, true, false, true>(ta, tb, to, p, m_tiles, st);
    if (p.ep.act == SBGM_ACT_GELU) return launch_conv_tc_inst<FMT, BN, kStages, SBGM_ACT_GELU, 0, true, false, true>(ta, tb, to, p, m_tiles, st);
    set_error("conv2d_tc: LayerNorm-folded Linear supports no activation or GELU");
    return 1;
  }
  if (p.ep.proj_w) {
    if (BLOCK_N != 64) { set_error("conv2d_tc: projection epilogue needs a 64-wide tile"); return 1; }
    return launch_conv_tc_inst<FMT, 64, (FMT == SBGM_FMT_BF16X2 ? 2 : 4), SBGM_ACT_NONE, 1, false>(ta, tb, to, p, m_tiles, st);
  }
  if (p.ep.staged) {
    if constexpr (TcFmt<FMT>::kAPlanes == 1 && BLOCK_N <= 128) {
      if (p.mt == 2) {       // two pixel tiles per CTA: 2 x 16 KB of A + the weight boxes per stage
        constexpr int kS2 = (TcFmt<FMT>::kBPlanes == 2 && BLOCK_N == 128) ? 3 : 4;
        SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kS2, ACT, 0, true, false, false, 2>(ta, tb, to, p, m_tiles, st)));
      }
    }
    SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kStages, ACT, 0, true>(ta, tb, to, p, m_tiles, st)));
  }
  SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kStages, ACT, 0, false>(ta, tb, to, p, m_tiles, st)));
  return 0;
}

// slab mode: staged TMA-store epilogue only, four weight stages
template <int FMT, int BLOCK_N>
static int launch_conv_tc_slab(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const ConvTcParams& p, int m_tiles,
                               cudaStream_t st) {
  constexpr int kBStages = (FMT == SBGM_FMT_BF16X2 && BLOCK_N == 128) ? 3 : 4;     // 2 x 50 KB of slabs + 3 x 32 KB of weights
  if (p.ep.staged) {
    if constexpr (TcFmt<FMT>::kAPlanes == 1 && BLOCK_N <= 128) {
      if (p.mt == 2) {       // two halo slabs per A stage (2 x 2 x 25.6 KB) + the weight ring
        constexpr int kS2 = (TcFmt<FMT>::kBPlanes == 2 && BLOCK_N == 128) ? 3 : 4;
        if (p.cluster == 2)
          SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kS2, ACT, 0, true, true, false, 2, 2>(ta, tb, to, p, m_tiles, st)));
        SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kS2, ACT, 0, true, true, false, 2>(ta, tb, to, p, m_tiles, st)));
      }
      if (p.cluster == 2)
        SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kBStages, ACT, 0, true, true, false, 1, 2>(ta, tb, to, p, m_tiles, st)));
    }
    SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kBStages, ACT, 0, true, true>(ta, tb, to, p, m_tiles, st)));
  }
  SBGM_DISPATCH_ACT(p.ep.act, return (launch_conv_tc_inst<FMT, BLOCK_N, kBStages, ACT, 0, false, true>(ta, tb, to, p, m_tiles, st)));
  return 0;
}

}  // namespace sbgm

using namespace sbgm;

// Split-K factor: layers whose output grid leaves most SMs idle and whose K loop is long (the 4x4 / 8x8 maps)
// are bound by one SM's operand ingest; slicing K over up to 4 CTAs spreads the same bytes over 4x the SMs.
static int pick_splits(int ctas, int total_kb) {
  int splits = 1;
  while (splits < 4 && ctas * splits * 2 <= 148 && total_kb / (splits * 2) >= 8) splits *= 2;
  return splits;
}

static void conv_tc_geometry(int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, int planes,
                             ConvTcParams* p, int* block_n, int* m_tiles, int ho_override = 0, int wo_override = 0) {
  p->n = n;
  p->ho = ho_override > 0 ? ho_override : (h + 2 * pad - kh) / stride + 1;
  p->wo = wo_override > 0 ? wo_override : (w + 2 * pad - kw) / stride + 1;
  p->kh = kh; p->kw = kw; p->stride = stride; p->pad_h = pad; p->pad_w = pad;
  p->out_h = p->ho; p->out_w = p->wo; p->out_step = 1; p->out_oy = 0; p->out_ox = 0;
  pick_tile(n, p->ho, p->wo, &p->w_tile, &p->h_tile, &p->n_tile);
  p->tiles_w = ceil_div(p->wo, p->w_tile);
  p->tiles_h = ceil_div(p->ho, p->h_tile);
  p->cin_blocks = cin / 64;
  p->slab_perm = 0; p->slab_row = 0; p->slab_tx = 0;
  *m_tiles = p->tiles_w * p->tiles_h * ceil_div(n, p->n_tile);
  *block_n = (cout % 256 == 0 && planes == 1) ? 256 : (cout % 128 == 0 ? 128 : 64);
  // under-filled grids (the attention blocks' Linear layers): narrower tiles = more CTAs and a shorter epilogue each
  // (short K loops only: with a long K loop the narrower tile re-reads the activation tile more often than it saves)
  while (*block_n > 64 && kh * kw * p->cin_blocks <= 8 && static_cast<long long>(*m_tiles) * (cout / *block_n) * 2 <= 148) *block_n /= 2;
  p->splits = pick_splits(*m_tiles * (cout / *block_n), kh * kw * p->cin_blocks);
}

// chunks per image of the fused GroupNorm statistics, or 0 if this shape cannot fuse them
static int gn_chunks_for(const ConvTcParams& p) {
  if (p.splits > 1) return 0;
  if (p.n_tile == 1) return p.tiles_w * p.tiles_h * 4;
  const int hw = p.ho * p.wo;
  if (p.h_tile == p.ho && p.w_tile == p.wo && hw % 32 == 0) return hw / 32;
  return 0;
}

extern "C" int sbgm_conv2d_tc_gn_chunks(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad) {
  if (cin % 64 != 0 || cout % 64 != 0 || stride < 1) return 0;
  ConvTcParams p;
  int block_n = 0, m_tiles = 0;
  conv_tc_geometry(n, h, w, cin, cout, kh, kw, stride, pad, fmt == SBGM_FMT_BF16 ? 1 : 2, &p, &block_n, &m_tiles);
  if (p.ho <= 0 || p.wo <= 0) return 0;
  return gn_chunks_for(p);
}

extern "C" size_t sbgm_conv2d_tc_workspace_bytes(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw,
                                                 int stride, int pad) {
  if (cin % 64 != 0 || cout % 64 != 0 || stride < 1) return 0;
  ConvTcParams p;
  int block_n = 0, m_tiles = 0;
  conv_tc_geometry(n, h, w, cin, cout, kh, kw, stride, pad, fmt == SBGM_FMT_BF16 ? 1 : 2, &p, &block_n, &m_tiles);
  if (p.ho <= 0 || p.wo <= 0 || p.splits <= 1) return 0;
  return static_cast<size_t>(p.splits) * n * p.ho * p.wo * cout * sizeof(float);
}

struct ConvTcEx {      // optional generalisation used by the data-gradient path (all zero = plain convolution)
  int pad_h, pad_w, ho, wo, out_h, out_w, out_step, out_oy, out_ox, res_pix_mod;
  bool on;
};

static int conv2d_tc_impl(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                          const void* residual, size_t res_plane, const float* tproj, int tproj_stride,
                          void* out, size_t out_plane, int fmt, int n, int h, int w, int cin, int cout,
                          int kh, int kw, int stride, int pad, int act, const float* proj_w, int n_proj,
                          float* proj_out, void* workspace, size_t workspace_bytes, float* gn_partials,
                          const ConvTcEx& ex, void* stream, const float* ln_colsum = nullptr, float ln_eps = 0.0f) {
  SBGM_REQUIRE(fmt == SBGM_FMT_BF16 || fmt == SBGM_FMT_BF16X2 || fmt == SBGM_FMT_F16, "conv2d_tc: format %d is not a tensor-core format", fmt);
  SBGM_REQUIRE(cin % 64 == 0 && cout % 64 == 0, "conv2d_tc: cin=%d and cout=%d must be multiples of 64", cin, cout);
  SBGM_REQUIRE(stride >= 1 && stride <= 8, "conv2d_tc: stride %d unsupported", stride);
  SBGM_REQUIRE(proj_w == nullptr || (cout == 64 && n_proj == kProjN && proj_out != nullptr && residual == nullptr &&
                                     tproj == nullptr && act == SBGM_ACT_NONE),
               "conv2d_tc: the projection epilogue needs cout == 64, n_proj == %d and a bias-only epilogue", kProjN);
  const int ho = ex.on ? ex.ho : (h + 2 * pad - kh) / stride + 1, wo = ex.on ? ex.wo : (w + 2 * pad - kw) / stride + 1;
  SBGM_REQUIRE(ho > 0 && wo > 0, "conv2d_tc: empty output");
  const int planes = (fmt == SBGM_FMT_BF16X2) ? 2 : 1;        // activation planes
  const int w_planes = (fmt == SBGM_FMT_BF16) ? 1 : 2;        // weight planes (hi | lo)

  ConvTcParams p;
  int block_n = 0, m_tiles = 0;
  conv_tc_geometry(n, h, w, cin, cout, kh, kw, stride, pad, w_planes, &p, &block_n, &m_tiles, ex.on ? ex.ho : 0, ex.on ? ex.wo : 0);
  bool scatter = false;
  if (ex.on) {
    p.pad_h = ex.pad_h; p.pad_w = ex.pad_w;
    p.out_h = ex.out_h; p.out_w = ex.out_w; p.out_step = ex.out_step; p.out_oy = ex.out_oy; p.out_ox = ex.out_ox;
    scatter = !(ex.out_step == 1 && ex.out_oy == 0 && ex.out_ox == 0 && ex.out_h == ho && ex.out_w == wo);
    SBGM_REQUIRE((ho - 1) * ex.out_step + ex.out_oy < ex.out_h && (wo - 1) * ex.out_step + ex.out_ox < ex.out_w,
                 "conv2d_tc: scattered output exceeds the output tensor");
    SBGM_REQUIRE(proj_w == nullptr && gn_partials == nullptr, "conv2d_tc: extended addressing excludes the projection / GroupNorm epilogues");
  }
  const size_t ws_need = static_cast<size_t>(p.splits) * n * ho * wo * cout * sizeof(float);
  if (p.splits > 1 && (scatter || proj_w != nullptr || workspace == nullptr || workspace_bytes < ws_need)) p.splits = 1;
  if (ln_colsum != nullptr) {
    SBGM_REQUIRE(kh == 1 && kw == 1 && stride == 1 && !ex.on && proj_w == nullptr && gn_partials == nullptr && out != nullptr,
                 "conv2d_tc: the LayerNorm fold applies to plain Linear layers");
    p.splits = 1;
    if (block_n > 128) block_n = 128;
  }
  p.ln_colsum = ln_colsum;
  p.ln_eps = ln_eps;
  p.ws = static_cast<float*>(workspace);
  p.gn_partials = gn_partials;
  p.gn_chunks = gn_chunks_for(p);
  SBGM_REQUIRE(gn_partials == nullptr || (p.gn_chunks > 0 && residual == nullptr && tproj == nullptr && act == SBGM_ACT_NONE &&
                                          proj_w == nullptr),
               "conv2d_tc: this shape / epilogue cannot fuse GroupNorm statistics (query sbgm_conv2d_tc_gn_chunks first)");
  p.ep.bias = bias; p.ep.residual = residual; p.ep.res_plane = res_plane; p.ep.res_pix_mod = ex.on ? ex.res_pix_mod : 0; p.ep.tproj = tproj; p.ep.tproj_stride = tproj_stride;
  p.ep.act = act; p.ep.cout = cout; p.ep.out = out; p.ep.out_plane = out_plane;
  p.ep.proj_w = proj_w; p.ep.proj_out = proj_out; p.ep.n_proj = n_proj;
  SBGM_REQUIRE(p.w_tile * stride <= 256 && p.h_tile * stride <= 256, "conv2d_tc: TMA box too large for stride %d", stride);

  // dense output addressing, full epilogue: the tile leaves through shared memory and TMA stores
  p.ep.staged = (!scatter && proj_w == nullptr && p.splits == 1 && out != nullptr) ? 1 : 0;
  // 3x3 / stride 1 / pad 1: one halo slab per 64-channel block.  Maps tileable by 16 rows x 8 columns
  // use 16 x 8 tiles of one image; other maps tileable by 8 x 8 use 8 x 8 tiles of two images with permuted tensor maps
  // (no fused GroupNorm statistics there: a warp's 32 rows span two images).  Split-K slices the 64-channel blocks.
  bool slab = (p.ep.staged || (p.splits > 1 && proj_w == nullptr && !scatter)) && kh == 3 && kw == 3 && stride == 1 &&
              p.pad_h == 1 && p.pad_w == 1 && ho == h && wo == w && wo % 8 == 0 && ho % 8 == 0;
  const bool slab_perm = slab && ho % kSlabTileH != 0;
  if (slab_perm && gn_partials != nullptr) slab = false;
  if (slab && p.splits > 1 && (p.splits - 1) * ceil_div(p.cin_blocks, p.splits) >= p.cin_blocks) slab = false;
  // slab mode makes the activation operand cheap to re-read: a two-way split-K 128-wide layer (the 8 x 8 maps) runs instead as
  // twice as many 64-wide tiles over the whole K loop -- same CTA count, no partial tiles, no finalize kernel
  if (slab && p.splits == 2 && block_n == 128 && out != nullptr) {
    block_n = 64;
    p.splits = 1;
    p.ep.staged = 1;
  }
  if (slab) {
    p.slab_perm = slab_perm ? 1 : 0;
    p.w_tile = 8; p.h_tile = slab_perm ? 8 : 16; p.n_tile = slab_perm ? 2 : 1;
    p.tiles_w = wo / 8; p.tiles_h = ho / p.h_tile;
    m_tiles = p.tiles_w * p.tiles_h * ceil_div(n, p.n_tile);
    p.slab_row = (slab_perm ? 2 : 1) * kSlabW * 8;
    p.slab_tx = (slab_perm ? 10 * 2 * 10 : kSlabW * kSlabH) * 128;
    if (!slab_perm) p.gn_chunks = gn_chunks_for(p);
  }
  // Two pixel tiles per CTA (MT = 2) where the grid stays full (>= 1.7 waves of one-tile CTAs): the weight boxes -- most of a
  // K-heavy layer's operand bytes -- are fetched once for both.  Measured per layer (profiles/r02_conv_tc_family_table_*.txt):
  // conv2 110 -> 66 us, 128->128 at 32 x 32 47 -> 42 us; trading a 128-wide one-wave grid for 64-wide two-tile CTAs was slower.
  p.mt = 1;
  {
    const bool allowed = planes == 1 && p.ep.staged && proj_w == nullptr && p.splits == 1 && ln_colsum == nullptr && block_n <= 128 &&
                         m_tiles >= 2;
    const long long ctas = static_cast<long long>(m_tiles) * (cout / block_n);
    if (allowed && ctas >= 252) p.mt = 2;
  }
  // Weight multicast over a CTA pair (CL = 2) in slab mode: both CTAs stream the same weight boxes (same output-channel block,
  // same K range), each loads half and multicasts it.  Single-plane activations, staged store, at least one full pair of CTAs
  // along the pixel tiles.  Measured per layer on the C2 forward (profiles/r02_conv_tc_family_table_fp16x2_cluster.txt against
  // ..._mt2_first.txt): the pair runs in lock step, so it pays only where the weight stream is what the layer waits for --
  // 512 -> 512 at 8 x 8: 40.4 -> 36.6 us (478 -> 528 TFLOP/s); the 128- and 256-channel layers are within +-1.5 us either way
  // (sum over the family 551.6 -> 555.7 us with the pair everywhere).  Hence pairs for cin, cout >= 512 only.
  p.cluster = 1;
  {
    const int ctas_x = (m_tiles + p.mt - 1) / p.mt;
    const bool allowed = slab && planes == 1 && p.ep.staged && proj_w == nullptr && ln_colsum == nullptr && block_n <= 128 && ctas_x >= 2;
    if (allowed && cin >= 512 && cout >= 512) p.cluster = 2;
  }
  CUtensorMap ta, tb, to;
  if (slab ? (slab_perm ? encode_perm_map(&ta, in, planes, in_plane, n, h, w, cin, kSlabW, 2, 10)
                        : encode_act_map(&ta, in, planes, in_plane, n, h, w, cin, kSlabW, kSlabH, 1, 1))
           : encode_act_map(&ta, in, planes, in_plane, n, h, w, cin, p.w_tile, p.h_tile, p.n_tile, stride)) return 1;
  const int K = kh * kw * cin;
  if (encode_weight_map(&tb, weight, w_planes, w_plane, cout, K, block_n / p.cluster)) return 1;     // a pair's CTA loads half the rows
  if (p.ep.staged) {
    if (slab && slab_perm ? encode_perm_map(&to, out, planes, out_plane, n, ho, wo, cout, 8, 2, 2)
                          : encode_out_map(&to, out, planes, out_plane, n, ho, wo, cout, p.w_tile, p.h_tile, p.n_tile)) return 1;
  } else {
    to = ta;
  }
  cudaStream_t st = as_stream(stream);
  if (slab) {
    if (fmt == SBGM_FMT_BF16) {
      if (block_n == 256) return launch_conv_tc_slab<SBGM_FMT_BF16, 256>(ta, tb, to, p, m_tiles, st);
      if (block_n == 128) return launch_conv_tc_slab<SBGM_FMT_BF16, 128>(ta, tb, to, p, m_tiles, st);
      return launch_conv_tc_slab<SBGM_FMT_BF16, 64>(ta, tb, to, p, m_tiles, st);
    }
    if (fmt == SBGM_FMT_F16) {
      if (block_n == 128) return launch_conv_tc_slab<SBGM_FMT_F16, 128>(ta, tb, to, p, m_tiles, st);
      return launch_conv_tc_slab<SBGM_FMT_F16, 64>(ta, tb, to, p, m_tiles, st);
    }
    if (block_n == 128) return launch_conv_tc_slab<SBGM_FMT_BF16X2, 128>(ta, tb, to, p, m_tiles, st);
    return launch_conv_tc_slab<SBGM_FMT_BF16X2, 64>(ta, tb, to, p, m_tiles, st);
  }
  if (fmt == SBGM_FMT_BF16) {
    if (block_n == 256) return launch_conv_tc<SBGM_FMT_BF16, 256, 4>(ta, tb, to, p, m_tiles, st);
    if (block_n == 128) return launch_conv_tc<SBGM_FMT_BF16, 128, 3>(ta, tb, to, p, m_tiles, st);
    return launch_conv_tc<SBGM_FMT_BF16, 64, 4>(ta, tb, to, p, m_tiles, st);
  }
  if (fmt == SBGM_FMT_F16) {      // one activation plane + two weight planes per stage: 48 KB (N = 128) / 32 KB (N = 64)
    if (block_n == 128) return launch_conv_tc<SBGM_FMT_F16, 128, 4>(ta, tb, to, p, m_tiles, st);
    return launch_conv_tc<SBGM_FMT_F16, 64, 4>(ta, tb, to, p, m_tiles, st);
  }
  if (block_n == 128) return launch_conv_tc<SBGM_FMT_BF16X2, 128, 3>(ta, tb, to, p, m_tiles, st);
  // short K loop on a grid of at most one CTA per SM (the attention blocks' Linear layers): four stages put the whole K loop
  // in flight at once -- one TMA round trip instead of two
  if (proj_w == nullptr && kh * kw * p.cin_blocks <= 8 && static_cast<long long>(m_tiles) * (cout / 64) * p.splits <= 148)
    return launch_conv_tc<SBGM_FMT_BF16X2, 64, 4>(ta, tb, to, p, m_tiles, st);
  return launch_conv_tc<SBGM_FMT_BF16X2, 64, 2>(ta, tb, to, p, m_tiles, st);
}

extern "C" int sbgm_conv2d_tc(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                              const void* residual, size_t res_plane, const float* tproj, int tproj_stride,
                              void* out, size_t out_plane, int fmt, int n, int h, int w, int cin, int cout,
                              int kh, int kw, int stride, int pad, int act, const float* proj_w, int n_proj,
                              float* proj_out, void* workspace, size_t workspace_bytes, float* gn_partials,
                              void* stream) {
  ConvTcEx ex = {};
  return conv2d_tc_impl(in, in_plane, weight, w_plane, bias, residual, res_plane, tproj, tproj_stride, out, out_plane, fmt, n, h, w,
                        cin, cout, kh, kw, stride, pad, act, proj_w, n_proj, proj_out, workspace, workspace_bytes, gn_partials, ex, stream);
}

// Generalised form used by the data gradients, the transposed-convolution decoder and the im2col stem: separate
// vertical / horizontal padding, an explicit logical output size (ho, wo), a scattered store
// out[n][oy * out_step + out_oy][ox * out_step + out_ox] into an [n][out_h][out_w][cout] tensor (`residual`, if given,
// is read at the same positions; res_pix_mod > 0 broadcasts a one-image residual over the batch).
extern "C" int sbgm_conv2d_tc_ex(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                                 const void* residual, size_t res_plane, int res_pix_mod, const float* tproj, int tproj_stride,
                                 void* out, size_t out_plane, int fmt, int n, int h,
                                 int w, int cin, int cout, int kh, int kw, int stride, int pad_h, int pad_w, int ho, int wo,
                                 int out_h, int out_w, int out_step, int out_oy, int out_ox, int act, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  ConvTcEx ex = {pad_h, pad_w, ho, wo, out_h, out_w, out_step, out_oy, out_ox, res_pix_mod, true};
  return conv2d_tc_impl(in, in_plane, weight, w_plane, bias, residual, res_plane, tproj, tproj_stride, out, out_plane, fmt, n, h, w, cin,
                        cout, kh, kw, stride, pad_h, act, nullptr, 0, nullptr, workspace, workspace_bytes, nullptr, ex, stream);
}

// y = act( LayerNorm(x; gamma, beta, eps) W^T + b ) over token rows x[rows][cin] -> y[rows][cout] with the LayerNorm folded into the
// GEMM (ImageSelfAttention: ln1 -> mha.in_proj, ln2 -> ff.0 + GELU, score_unet.py:139-146): `weight` holds W diag(gamma),
// `bias` = b + W beta, `colsum[cout]` = row sums of the folded weight; the per-token mean / rstd are computed inside the kernel
// from the operand tiles, the normalised tensor never exists.
extern "C" int sbgm_linear_ln_tc(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                                 const float* colsum, float eps, void* out, size_t out_plane, int fmt, int rows, int cin, int cout,
                                 int act, void* stream) {
  SBGM_REQUIRE(colsum != nullptr && bias != nullptr, "linear_ln_tc: colsum and bias are required");
  ConvTcEx ex = {};
  return conv2d_tc_impl(in, in_plane, weight, w_plane, bias, nullptr, 0, nullptr, 0, out, out_plane, fmt, 1, 1, rows, cin, cout, 1, 1, 1, 0,
                        act, nullptr, 0, nullptr, nullptr, 0, nullptr, ex, stream, colsum, eps);
}
