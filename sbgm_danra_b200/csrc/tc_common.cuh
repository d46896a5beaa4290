// tc_common.cuh -- PTX wrappers (mbarrier, TMA, tcgen05, TMEM) and the shared epilogue of the
// tensor-core convolution kernels (conv_tc.cu, conv3x3_c64.cu).  sm_100a only.
#pragma once

#include <cuda.h>

#include "common.cuh"

namespace sbgm {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a TMA fault or a descriptor bug would otherwise hang the GPU until the watchdog.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (!done && spin > (1u << 26)) __trap();
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// the same box delivered to the same shared-memory offset of every CTA in `cta_mask` of the cluster; each destination CTA's
// barrier (same offset) receives the complete_tx
__device__ __forceinline__ void tma_load_3d_multicast(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// bulk tensor store shared -> global (the epilogue's staged tile), tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
      ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute/arch/mma_sm100_desc.hpp):
//   [0,14) start >> 4 | [16,30) LBO >> 4 (unused with swizzle: 1) | [32,46) SBO >> 4 (8 rows x 128 B = 1024)
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t addr) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D = f32 (bits 4-5 = 1), A / B format (bits 7-9 / 10-12: 0 = float16, 1 = bfloat16), both
// K-major, M = 128, N = n.
__device__ __forceinline__ constexpr uint32_t make_idesc(int n, bool half = false) {
  return (1u << 4) | (half ? 0u : ((1u << 7) | (1u << 10))) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// `desc_lo` is the low descriptor word ((smem_addr & 0x3FFFF) >> 4 | LBO 1 << 16); the high word for K-major
// SWIZZLE_128B tiles is the constant kDescHi (SBO = 1024 B, version 1).  Advancing an operand by `bytes` is a plain
// add of bytes >> 4 to the descriptor.
constexpr uint32_t kDescHi = 64u | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); }
// Single-thread issue path: the caller has already narrowed the warp to one elected lane (elect_one()), so the
// MMA needs no per-instruction election or predicate vote.  Descriptors are whole 64-bit values; advancing an
// operand is one 64-bit add of bytes >> 4 (the address field never carries out of its 14 bits inside one CTA's
// shared memory window).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\tselp.u32 %0, 1, 0, q;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_bf16_acc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.eq.u32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_first(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same offset in every CTA of `cta_mask` once the MMAs issued so far have retired
__device__ __forceinline__ void umma_commit_multicast(uint32_t bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot_smem_addr, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot_smem_addr), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- epilogue ----------------------------------------------------------------------------------
// v = acc + bias[co];  v += residual[pix][co];  v = act(v);  v += tproj[n][co];  store (NHWC, fmt)
// Projection mode (cout == 64 tiles, one thread holds a whole pixel): instead of storing the 64
// channels, accumulate kProjN dot products  proj[q] += sum_c v[c] * c_proj_w[q][c]  -- the nine taps of
// the final 64 -> 1 convolution (Decoder.final_layer.conv, score_unet.py:713-730) -- and store them
// as proj_out[pix][SBGM_PROJ_STRIDE] fp32.  The 9 x 64 weights live in constant memory so every FFMA
// takes its weight as a constant-bank operand (no loads, warp-uniform address).
struct EpilogueParams {
  const float* bias;
  const void* residual;
  size_t res_plane;
  int res_pix_mod;       // > 0: the residual is broadcast over the batch, indexed by pix % res_pix_mod
  const float* tproj;
  int tproj_stride;
  int act;
  int cout;
  void* out;
  size_t out_plane;
  int staged;            // 1: outputs leave through shared memory + TMA store (conv_tc.cu, dense output addressing)
  const float* proj_w;   // [kProjN][64] fp32 (device) or nullptr; copied to c_proj_w before the launch
  float* proj_out;       // [pix][SBGM_PROJ_STRIDE] fp32
  int n_proj;
};
constexpr int kProjN = 9;
constexpr int kProjMax = SBGM_PROJ_STRIDE;
static __constant__ __align__(16) float c_proj_w[kProjN * 64];

template <int ACT>
__device__ __forceinline__ float act_ct(float x) {
  if (ACT == SBGM_ACT_RELU) return fmaxf(x, 0.0f);
  if (ACT == SBGM_ACT_SILU) return silu(x);
  if (ACT == SBGM_ACT_GELU) return gelu_erf(x);
  return x;
}

// 8 x 8 transpose of 16-byte items inside each group of 8 lanes: on entry lane j of a group holds the 8
// channel-chunks of ITS pixel; on exit it holds chunk j of the group's 8 pixels, so that a group writes one
// full 128-byte line per store instruction (4 lines per warp-instruction instead of 32).
__device__ __forceinline__ void transpose8_u4(uint4 (&v)[8], int lane) {
#pragma unroll
  for (int s = 4; s >= 1; s >>= 1) {
    const bool up = (lane & s) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (i & s) continue;
      const uint4 send = up ? v[i] : v[i | s];
      uint4 recv;
      recv.x = __shfl_xor_sync(0xffffffffu, send.x, s);
      recv.y = __shfl_xor_sync(0xffffffffu, send.y, s);
      recv.z = __shfl_xor_sync(0xffffffffu, send.z, s);
      recv.w = __shfl_xor_sync(0xffffffffu, send.w, s);
      if (up) v[i] = recv; else v[i | s] = recv;
    }
  }
}

// Store one pixel's 64 consecutive channels (this lane's `v`) for all 32 lanes of the warp, coalesced through
// the 8-lane transpose.  Must be called by the whole warp; `valid` masks pixels outside the tensor.
template <int FMT>
__device__ __forceinline__ void store_block64(void* out, size_t out_plane, int cout, const float (&v)[64], size_t pix,
                                              bool valid, int co_base, int lane) {
  const int l8 = lane & 7, gbase = lane & ~7;
  constexpr int kPlanes = TcFmt<FMT>::kAPlanes;
#pragma unroll
  for (int pl = 0; pl < kPlanes; ++pl) {
    uint4 c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float t[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = v[j * 8 + e];
        t[e] = (pl == 0) ? x : x - bf16_round(x);
      }
      c[j] = TcFmt<FMT>::pack8(t);
    }
    // (256-bit stores of the lane's own row -- STG.256, one full sector per lane, no transpose, ~45 instead of ~270 instructions
    // per plane -- measured neutral in the sampler and 10 % slower on the fused conv_up: 32 distinct lines per instruction)
    transpose8_u4(c, lane);
    __nv_bfloat16* base = static_cast<__nv_bfloat16*>(out) + pl * out_plane;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const unsigned long long pk = __shfl_sync(0xffffffffu, static_cast<unsigned long long>(pix), gbase + k);
      const int vk = __shfl_sync(0xffffffffu, static_cast<int>(valid), gbase + k);
      if (vk) *reinterpret_cast<uint4*>(base + pk * cout + co_base + l8 * 8) = c[k];
    }
  }
}

// Staged variant: the lane's pixel row (64 channels = 128 bytes per plane) goes to shared memory in the 128-byte-swizzle
// layout of a TMA box (chunk j of row r at r * 128 + ((j ^ (r & 7)) << 4): conflict-free 16-byte stores), and one lane
// hands the warp's 32 x 64 sub-box to the TMA unit.  Replaces the shuffle transpose + 8 predicated stores per plane --
// ~220 of the ~270 instructions per plane in an epilogue that ncu showed to be the kernels' critical path; bounds clipping
// comes from the tensor map.  `stage` = this warp's staging area for this block (planes kStageBlockBytes apart).
constexpr uint32_t kStageBlockBytes = 32 * 128;
template <int FMT>
__device__ __forceinline__ void store_block64_staged(const CUtensorMap* tmap_o, uint32_t stage, const float (&v)[64], int co_base,
                                                     int x0, int y0, int n0, int lane) {
  constexpr int kPlanes = TcFmt<FMT>::kAPlanes;
#pragma unroll
  for (int pl = 0; pl < kPlanes; ++pl) {
    const uint32_t row = stage + pl * kStageBlockBytes + lane * 128;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float t[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float x = v[j * 8 + e];
        t[e] = (pl == 0) ? x : x - bf16_round(x);
      }
      const uint4 c = TcFmt<FMT>::pack8(t);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + ((j ^ (lane & 7)) << 4)), "r"(c.x), "r"(c.y), "r"(c.z), "r"(c.w) : "memory");
    }
  }
  fence_async_shared();
  __syncwarp();
  if (lane == 0) {
#pragma unroll
    for (int pl = 0; pl < kPlanes; ++pl) tma_store_5d(tmap_o, stage + pl * kStageBlockBytes, co_base, x0, y0, n0, pl);
    tma_store_commit();
  }
}

// Two fp32 operations per issue slot (FADD2 / FFMA2): the epilogue warps are issue-bound next to the MMA issuer.
__device__ __forceinline__ void add_f32x2(float& a0, float& a1, float b0, float b1) {
  unsigned long long a, b;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(a) : "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(a));
}
// (a0, a1) += s * (t0, t1)
__device__ __forceinline__ void fma_scalar_f32x2(float& a0, float& a1, float t0, float t1, float s) {
  unsigned long long a, t, ss;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(t) : "f"(t0), "f"(t1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(ss) : "f"(s));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a) : "l"(t), "l"(ss));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(a));
}

// GroupNorm partial statistics of one 64-channel block, at 8-channel granularity, reduced over the warp's 32
// rows: dst[sub][2] (sum, sum of squares) for sub = 0..7.  Values are taken as stored (bias added, bf16-rounded
// in the single-plane modes).  Must be called by the whole warp; rows with !valid contribute nothing.
template <int FMT>
__device__ __forceinline__ void gn_block64_stats(const uint32_t (&ra)[32], const uint32_t (&rb)[32], const float* bias,
                                                 int co_base, bool valid, int lane, float* dst) {
  // x[2 g] = sum, x[2 g + 1] = sum of squares of group g over this thread's row (packed fp32: two channels per instruction)
  float x[16];
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __uint_as_float(g < 4 ? ra[g * 8 + j] : rb[(g - 4) * 8 + j]);
    if (bias) {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + co_base + g * 8)), b1 = __ldg(reinterpret_cast<const float4*>(bias + co_base + g * 8) + 1);
      add_f32x2(v[0], v[1], b0.x, b0.y);
      add_f32x2(v[2], v[3], b0.z, b0.w);
      add_f32x2(v[4], v[5], b1.x, b1.y);
      add_f32x2(v[6], v[7], b1.z, b1.w);
    }
    if (FMT == SBGM_FMT_BF16 || FMT == SBGM_FMT_F16) {      // the statistics describe the values as stored
#pragma unroll
      for (int j = 0; j < 8; j += 2) TcFmt<FMT>::round2(v[j], v[j + 1]);
    }
    if (!valid) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.0f;
    }
    unsigned long long p[4], sp, qp;
#pragma unroll
    for (int j = 0; j < 4; ++j) asm("mov.b64 %0, {%1, %2};" : "=l"(p[j]) : "f"(v[2 * j]), "f"(v[2 * j + 1]));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(sp) : "l"(p[0]), "l"(p[1]));
    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(qp) : "l"(p[0]));
#pragma unroll
    for (int j = 1; j < 4; ++j) {
      if (j > 1) asm("add.rn.f32x2 %0, %0, %1;" : "+l"(sp) : "l"(p[j]));
      asm("fma.rn.f32x2 %0, %1, %1, %0;" : "+l"(qp) : "l"(p[j]));
    }
    float s0, s1, q0, q1;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(sp));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(q0), "=f"(q1) : "l"(qp));
    x[2 * g] = s0 + s1;
    x[2 * g + 1] = q0 + q1;
  }
  // transposing butterfly over the warp's 32 rows: each step halves the values a lane carries (16 shuffles instead of 80);
  // after the steps 16, 8, 4, 2 lane L holds value ((L >> 4) & 1) * 8 + ((L >> 3) & 1) * 4 + ((L >> 2) & 1) * 2 + ((L >> 1) & 1)
#pragma unroll
  for (int step = 0; step < 4; ++step) {
    const int off = 16 >> step, cnt = 8 >> step;
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < cnt; ++i) {
      const float send = upper ? x[i] : x[i + cnt], keep = upper ? x[i + cnt] : x[i];
      x[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  x[0] += __shfl_xor_sync(0xffffffffu, x[0], 1);
  if ((lane & 1) == 0) dst[((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1)] = x[0];
}

// 64 accumulator columns (two 32-column TMEM loads) of one row.  ACT and PROJ are compile-time
// (PROJ: 0 = store, 1 = projection only, 2 = projection AND store -- the training forward keeps the tensor).
struct StageArgs {          // where a staged block goes (unused when !STAGED)
  const CUtensorMap* tmap_o;
  uint32_t stage;
  int x0, y0, n0;
};

// acc += lo * kLoScale for the x * w_lo half of the accumulator, two columns per instruction
template <int FMT>
__device__ __forceinline__ void merge_lo(uint32_t (&r)[32], const uint32_t (&t)[32]) {
#pragma unroll
  for (int j = 0; j < 32; j += 2) {
    float a0 = __uint_as_float(r[j]), a1 = __uint_as_float(r[j + 1]);
    fma_scalar_f32x2(a0, a1, __uint_as_float(t[j]), __uint_as_float(t[j + 1]), TcFmt<FMT>::kLoScale);
    r[j] = __float_as_uint(a0);
    r[j + 1] = __float_as_uint(a1);
  }
}

template <int FMT, int ACT, int PROJ, bool STAGED = false>
__device__ __forceinline__ void epilogue_block64(const EpilogueParams& ep, const uint32_t (&ra)[32], const uint32_t (&rb)[32],
                                                 int co_base, int n, size_t pix, bool valid, int lane,
                                                 float (&proj_acc)[kProjMax], const StageArgs& sa = StageArgs{}) {
  float v[64];
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    v[j] = __uint_as_float(ra[j]);
    v[32 + j] = __uint_as_float(rb[j]);
  }
  if (ep.bias) {
#pragma unroll
    for (int g = 0; g < 16; ++g) {
      const float4 b = __ldg(reinterpret_cast<const float4*>(ep.bias + co_base) + g);
      add_f32x2(v[4 * g], v[4 * g + 1], b.x, b.y);
      add_f32x2(v[4 * g + 2], v[4 * g + 3], b.z, b.w);
    }
  }
  if (!PROJ && ep.residual && valid) {
#pragma unroll
    for (int g = 0; g < 8; ++g) {
      float rv[8];
      Act<FMT>::load8(ep.residual, ep.res_plane, (ep.res_pix_mod ? pix % ep.res_pix_mod : pix) * ep.cout + co_base + g * 8, rv);
#pragma unroll
      for (int j = 0; j < 8; j += 2) add_f32x2(v[g * 8 + j], v[g * 8 + j + 1], rv[j], rv[j + 1]);
    }
  }
#pragma unroll
  for (int j = 0; j < 64; ++j) v[j] = act_ct<ACT>(v[j]);
  if (!PROJ && ep.tproj && valid) {
    const float4* tp = reinterpret_cast<const float4*>(ep.tproj + static_cast<size_t>(n) * ep.tproj_stride + co_base);
#pragma unroll
    for (int g = 0; g < 16; ++g) {
      const float4 t = __ldg(tp + g);
      add_f32x2(v[4 * g], v[4 * g + 1], t.x, t.y);
      add_f32x2(v[4 * g + 2], v[4 * g + 3], t.z, t.w);
    }
  }
  if (PROJ) {
    // two channels per instruction (FFMA2, the weight pair straight from the constant bank): 288 instead of 576 issue slots per
    // pixel -- the epilogue warps share their schedulers with the MMA issuer and, in the fused-upsample kernel, the producers.
    // Each tap keeps an (even channels, odd channels) pair of partial sums, added at the end.
    unsigned long long acc2[kProjN];
#pragma unroll
    for (int q = 0; q < kProjN; ++q) acc2[q] = 0ull;
#pragma unroll
    for (int j = 0; j < 64; j += 2) {
      unsigned long long vp;
      asm("mov.b64 %0, {%1, %2};" : "=l"(vp) : "f"(v[j]), "f"(v[j + 1]));
#pragma unroll
      for (int q = 0; q < kProjN; ++q) {
        const unsigned long long wp = *reinterpret_cast<const unsigned long long*>(&c_proj_w[q * 64 + j]);
        asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc2[q]) : "l"(vp), "l"(wp));
      }
    }
#pragma unroll
    for (int q = 0; q < kProjN; ++q) {
      float lo, hi;
      asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(acc2[q]));
      proj_acc[q] += lo + hi;
    }
  }
  if (PROJ != 1) {          // PROJ == 2: both (training)
    if (STAGED) store_block64_staged<FMT>(sa.tmap_o, sa.stage, v, co_base, sa.x0, sa.y0, sa.n0, lane);
    else store_block64<FMT>(ep.out, ep.out_plane, ep.cout, v, pix, valid, co_base, lane);
  }
}

__device__ __forceinline__ void epilogue_store_proj(const EpilogueParams& ep, size_t pix, const float (&proj_acc)[kProjMax]) {
  float4* dst = reinterpret_cast<float4*>(ep.proj_out + pix * kProjMax);
  dst[0] = make_float4(proj_acc[0], proj_acc[1], proj_acc[2], proj_acc[3]);
  dst[1] = make_float4(proj_acc[4], proj_acc[5], proj_acc[6], proj_acc[7]);
  dst[2] = make_float4(proj_acc[8], proj_acc[9], proj_acc[10], proj_acc[11]);
}

// Runtime activation id -> compile-time template argument.
#define SBGM_DISPATCH_ACT(act, ...)                                                              \
  switch (act) {                                                                                  \
    case SBGM_ACT_NONE: { constexpr int ACT = SBGM_ACT_NONE; __VA_ARGS__; break; }                \
    case SBGM_ACT_RELU: { constexpr int ACT = SBGM_ACT_RELU; __VA_ARGS__; break; }                \
    case SBGM_ACT_GELU: { constexpr int ACT = SBGM_ACT_GELU; __VA_ARGS__; break; }                \
    case SBGM_ACT_SILU: { constexpr int ACT = SBGM_ACT_SILU; __VA_ARGS__; break; }                \
    default: ::sbgm::set_error("unknown activation %d", act); return 1;                            \
  }

// ---- host: tensor-map encoding -----------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_fn();
// NHWC activation [planes][n][h][w][c] bf16 as a 5-D map, box = (64, bw, bh, bn, 1), element strides (1, s, s, 1, 1)
int encode_act_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int n, int h, int w, int c,
                   int box_w, int box_h, int box_n, int stride, int box_c = 64);   // box_c = 32: 64-byte rows, SWIZZLE_64B
// NHWC output [planes][n][h][w][c] bf16 as a 5-D map whose box is a warp's 32-row share of a (box_w, box_h, box_n) tile
int encode_out_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int n, int h, int w, int c,
                   int tile_w, int tile_h, int tile_n);
// packed weights [planes][cout][K] bf16 as a 3-D map, box = (64, box_rows, 1)
int encode_weight_map(CUtensorMap* map, const void* base, int planes, size_t plane_elems, int cout, int K, int box_rows);
// (w_tile, h_tile, n_tile), product 128, powers of two, covering an [n][ho][wo] pixel grid with the least padding
void pick_tile(int n, int ho, int wo, int* wt, int* ht, int* nt);

}  // namespace sbgm
