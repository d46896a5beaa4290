// stem_dgrad_tc.cu -- data gradient of Encoder.conv1 (8x8, stride 2, pad 3; sbgm/score_unet.py:206-211, :312-315) on the
// tensor cores: from df = dL/d conv1(x || planes) [n][h/2][w/2][64] (activation format) to the fp32 NCHW gradients of x and of
// the conditioning planes.
//
// Input pixel (2 j + py, 2 i + px) only meets the taps r = 7 - py - 2 ky, s = 7 - px - 2 kx (ky, kx = 0..3), which read df at
// (j + py - 2 + ky, i + px - 2 + kx): each parity class (py, px) is a stride-1 4x4 convolution over df, an implicit GEMM with
// M = pixels of the class, N = cin padded to 16 (one tcgen05.mma N = 16 covers every input channel), K = 16 taps x 64.
//
// A CTA owns one class and walks tiles of 128 consecutive positions of the class grid, flattened row by row with each row padded
// to w/2 + 3 positions (two zero columns in front, one behind).  In that flattened layout a tap is a constant shift, and the
// columns a tap reads beyond either edge of a row are zero padding, so a tile's operand is one slab of df rows -- 128 + 3 (w/2 + 3)
// + 3 of them, written by the CTA's threads in the K-major 128-byte-swizzle layout -- and each tap's A operand is a descriptor
// start inside it (the slab addressing of conv_tc.cu).  The class's 16 x 1024 weights stay resident.  One elected lane issues
// the 64 (split-bf16: 128) MMAs of a tile; the 128 threads read one accumulator row each and store the class's pixels straight
// into dx / dplanes (fp32 NCHW).  Split bf16 (hi | lo planes): acc = a_hi (w_hi | w_lo) + a_lo w_hi, as the other kernels.
#include "tc_common.cuh"

namespace sbgm {

constexpr int kSdM = 128;              // class positions per tile
constexpr int kSdTaps = 16;            // 4 x 4 taps per class
constexpr int kSdN = 16;               // input channels, padded

struct StemDgradParams {
  const void* df;        // [n][hh][wh][64] in fmt
  size_t df_plane;
  const void* wt;        // [4 classes][planes][16][16 taps * 64] bf16 (sbgm_pack_weight, transposed, parity taps)
  size_t w_plane, w_class;
  float* dx;             // [n][1][h][w] or nullptr
  float* dpl;            // [n][cc][h][w] or nullptr
  int n, cc, h, w, hh, wh, wp;          // wp = wh + 3: padded row of the class grid
  int tiles_per_img, total_tiles, slab_rows;
  uint32_t slab_plane_bytes;
};

template <int FMT>
struct StemDgradCfg {
  static constexpr int kAPl = TcFmt<FMT>::kAPlanes, kBPl = TcFmt<FMT>::kBPlanes;
  static constexpr uint32_t kTapBytes = kBPl * kSdN * 128;          // one tap's B tile: [plane][16 ci][64 co]
  static constexpr uint32_t kWBytes = kSdTaps * kTapBytes;
  static constexpr uint32_t kSlabOffset = kWBytes;
  static uint32_t smem_bytes(uint32_t slab_plane_bytes) { return kSlabOffset + kAPl * slab_plane_bytes + 64 + 1024; }
};

template <int FMT>
__global__ void __launch_bounds__(128)
stem_dgrad_tc_kernel(const StemDgradParams p) {
  pdl_grid_sync();
  using Cfg = StemDgradCfg<FMT>;
  constexpr int kAPl = Cfg::kAPl, kBPl = Cfg::kBPl;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_base = smem_base, slab_base = smem_base + Cfg::kSlabOffset;
  const uint32_t bar_base = slab_base + kAPl * p.slab_plane_bytes;
  const uint32_t mma_bar = bar_base, tmem_slot = bar_base + 8;
  const uint32_t* tmem_slot_ptr = reinterpret_cast<const uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cls = blockIdx.y, py = cls >> 1, px = cls & 1;

  if (threadIdx.x == 0) {
    mbar_init(mma_bar, 1);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 32);

  // resident weights: tap t, row R = plane * 16 + ci, 16-byte chunk j (8 output channels of df)
  const __nv_bfloat16* wsrc = static_cast<const __nv_bfloat16*>(p.wt) + cls * p.w_class;
  for (int idx = threadIdx.x; idx < kSdTaps * kBPl * kSdN * 8; idx += blockDim.x) {
    const int j = idx & 7, R = (idx >> 3) % (kBPl * kSdN), t = idx / (8 * kBPl * kSdN);
    const int pl = R / kSdN, row = R % kSdN;
    const uint4 v = __ldg(reinterpret_cast<const uint4*>(wsrc + pl * p.w_plane + static_cast<size_t>(row) * (kSdTaps * 64) + t * 64 + j * 8));
    const uint32_t dst = w_base + t * Cfg::kTapBytes + R * 128 + ((j ^ (R & 7)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
  }

  const int omin = (py - 2) * p.wp + (px - 2);            // flattened offset of tap (0, 0)
  const size_t hw = static_cast<size_t>(p.h) * p.w;
  uint32_t it = 0;
  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x, ++it) {
    const int img = tile / p.tiles_per_img, q0 = (tile % p.tiles_per_img) * kSdM;
    // ---- slab: row s holds df at class-grid position q0 + omin + s (zero outside the map and in the padding columns) ----
    const uint8_t* dfi = static_cast<const uint8_t*>(p.df) + static_cast<size_t>(img) * p.hh * p.wh * 128;
    for (int idx = threadIdx.x; idx < p.slab_rows * 8; idx += blockDim.x) {
      const int s = idx >> 3, j = idx & 7;
      const int q = q0 + omin + s;
      const int jy = q >= 0 ? q / p.wp : -((p.wp - 1 - q) / p.wp);
      const int jx = q - jy * p.wp - 2;
      const bool in = jy >= 0 && jy < p.hh && jx >= 0 && jx < p.wh;
      const uint32_t dst = slab_base + s * 128 + ((j ^ (s & 7)) << 4);
#pragma unroll
      for (int pl = 0; pl < kAPl; ++pl) {
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (in) v = __ldg(reinterpret_cast<const uint4*>(dfi + pl * p.df_plane * 2 + (static_cast<size_t>(jy) * p.wh + jx) * 128) + j);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst + pl * p.slab_plane_bytes), "r"(v.x), "r"(v.y), "r"(v.z),
                     "r"(v.w) : "memory");
      }
    }
    fence_async_shared();             // generic-proxy stores -> visible to the tensor cores
    tcgen05_fence_before();
    __syncthreads();                  // slab and weights complete; the previous tile's accumulator has been read
    tcgen05_fence_after();
    const uint32_t tmem_d = *tmem_slot_ptr;
    if (warp == 0) {
      if (elect_one()) {
        constexpr uint32_t idesc_hi = make_idesc(kSdN * kBPl), idesc_lo = make_idesc(kSdN);
        const uint64_t a0 = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo(slab_base);
        const uint64_t b0 = (static_cast<uint64_t>(kDescHi) << 32) | desc_lo(w_base);
#pragma unroll 1
        for (int t = 0; t < kSdTaps; ++t) {
          const uint64_t a = a0 + static_cast<uint32_t>(((t >> 2) * p.wp + (t & 3)) * 8);   // 128-byte rows = 8 descriptor units
          const uint64_t b = b0 + t * (Cfg::kTapBytes >> 4);
#pragma unroll
          for (int k = 0; k < 4; ++k) {                                                  // K = 16 channels = 32 bytes per MMA
            umma_bf16(tmem_d, a + 2 * k, b + 2 * k, idesc_hi, (t | k) != 0);
            if (kAPl == 2) umma_bf16_acc(tmem_d, a + (p.slab_plane_bytes >> 4) + 2 * k, b + 2 * k, idesc_lo);
          }
        }
        umma_commit(mma_bar);
      }
      __syncwarp();
    }
    mbar_wait(mma_bar, it & 1u);
    tcgen05_fence_after();
    uint32_t r[32];
    tmem_ld32(tmem_d + (static_cast<uint32_t>(warp * 32) << 16), r);
    // ---- epilogue: accumulator row m = class-grid position q0 + m -> input pixel (2 jy + py, 2 jx + px) ----
    const int q = q0 + warp * 32 + lane;
    const int jy = q / p.wp, jx = q - jy * p.wp - 2;
    if (jy < p.hh && jx >= 0 && jx < p.wh) {
      const size_t pix = static_cast<size_t>(2 * jy + py) * p.w + 2 * jx + px;
      float v[kSdN];
#pragma unroll
      for (int c = 0; c < kSdN; ++c) v[c] = __uint_as_float(r[c]) + (kBPl == 2 ? __uint_as_float(r[kSdN + c]) * TcFmt<FMT>::kLoScale : 0.0f);
      if (p.dx) p.dx[img * hw + pix] = v[0];
      if (p.dpl) {
        float* d = p.dpl + static_cast<size_t>(img) * p.cc * hw + pix;
#pragma unroll
        for (int c = 1; c < kSdN; ++c)
          if (c <= p.cc) d[(c - 1) * hw] = v[c];
      }
    }
    tcgen05_fence_before();
  }
  __syncthreads();
  if (warp == 0) tmem_dealloc(*tmem_slot_ptr, 32);
}

template <int FMT>
static int launch_stem_dgrad_tc(const StemDgradParams& p, cudaStream_t st) {
  using Cfg = StemDgradCfg<FMT>;
  auto kern = stem_dgrad_tc_kernel<FMT>;
  const uint32_t smem = Cfg::smem_bytes(p.slab_plane_bytes);
  int dev = 0, max_smem = 0, num_sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
  SBGM_REQUIRE(smem <= static_cast<uint32_t>(max_smem), "stem_dgrad_tc: w=%d needs %u bytes of shared memory per CTA (at most %d)", p.w,
               smem, max_smem);
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) {
    set_error("stem_dgrad_tc: cannot reserve %u bytes of shared memory", smem);
    return 1;
  }
  const int per_sm = resident_blocks(reinterpret_cast<const void*>(kern), 128, smem) / (num_sms > 0 ? num_sms : 1);
  const int ctas = ceil_div(static_cast<long long>(num_sms) * (per_sm > 0 ? per_sm : 1), 4);
  launch_k((kern), dim3(p.total_tiles < ctas ? p.total_tiles : ctas, 4), 128, smem, st, p);
  return check_launch("stem_dgrad_tc");
}

}  // namespace sbgm

using namespace sbgm;

extern "C" int sbgm_stem_dgrad_tc(const void* df, size_t df_plane, int fmt, const void* w_packed, size_t w_plane, float* dx, float* dplanes,
                                  int np, int cc, int n, int h, int w, float* workspace, void* stream) {
  SBGM_REQUIRE(fmt == SBGM_FMT_BF16 || fmt == SBGM_FMT_BF16X2, "stem_dgrad_tc: format %d is not a bf16 training format", fmt);
  SBGM_REQUIRE(h % 2 == 0 && w % 2 == 0 && h > 0 && w > 0, "stem_dgrad_tc: h=%d and w=%d must be even", h, w);
  SBGM_REQUIRE(cc >= 0 && cc < kSdN, "stem_dgrad_tc: %d conditioning channels (at most %d)", cc, kSdN - 1);
  SBGM_REQUIRE(np == 1 || np == n, "stem_dgrad_tc: planes batch %d must be 1 or %d", np, n);
  SBGM_REQUIRE(dplanes == nullptr || (cc > 0 && (np == n || n == 1 || workspace != nullptr)),
               "stem_dgrad_tc: dplanes needs cc > 0 and, for planes shared by the batch, a workspace");
  StemDgradParams p;
  p.df = df; p.df_plane = df_plane; p.wt = w_packed; p.w_plane = w_plane; p.w_class = (fmt == SBGM_FMT_BF16X2 ? 2 : 1) * w_plane;
  p.dx = dx;
  const bool sum_batch = dplanes != nullptr && np == 1 && n > 1;
  p.dpl = sum_batch ? workspace : dplanes;
  p.n = n; p.cc = cc; p.h = h; p.w = w; p.hh = h / 2; p.wh = w / 2; p.wp = p.wh + 3;
  p.tiles_per_img = ceil_div(static_cast<long long>(p.hh) * p.wp, kSdM);
  p.total_tiles = p.tiles_per_img * n;
  p.slab_rows = kSdM + 3 * p.wp + 3;
  p.slab_plane_bytes = static_cast<uint32_t>((p.slab_rows + 7) / 8 * 8 * 128);
  SBGM_REQUIRE(w_plane >= static_cast<size_t>(kSdN) * kSdTaps * 64, "stem_dgrad_tc: weight plane of %zu elements is too small", w_plane);
  cudaStream_t st = as_stream(stream);
  const int rc = fmt == SBGM_FMT_BF16 ? launch_stem_dgrad_tc<SBGM_FMT_BF16>(p, st) : launch_stem_dgrad_tc<SBGM_FMT_BF16X2>(p, st);
  if (rc != 0 || !sum_batch) return rc;
  return stem_dgrad_batch_sum(workspace, dplanes, n, static_cast<size_t>(cc) * h * w, st);
}
