// common.cuh -- shared device/host helpers for the sbgm_b200 kernels (sm_100a).
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "../../include/sbgm_b200.h"

namespace sbgm {

// ---- host-side error plumbing --------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);   // cudaGetLastError -> status
#define SBGM_REQUIRE(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      ::sbgm::set_error(__VA_ARGS__);       \
      return 1;                             \
    }                                       \
  } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- launches: programmatic dependent launch (PDL) ------------------------------------------------------
// A sampler step is ~150 and a training step ~1 500 short kernels back to back on one stream (replayed from a
// CUDA graph).  Every kernel is launched with programmatic stream serialization and starts with pdl_grid_sync():
// it releases its own dependents at once and then waits for its predecessor to complete and flush, so the next
// kernel's blocks are scheduled (and its launch latency paid) while the previous grid drains.  Semantics are those
// of an ordinary in-order stream because no kernel touches global memory before the wait.
// SBGM_B200_PDL=0 disables the attribute (the device-side instructions are then no-ops).
void note_launch_error(cudaError_t e);
bool pdl_enabled();
int resident_blocks(const void* kern, int block, size_t smem);   // blocks of `kern` resident at once on the GPU (elementwise.cu)
// out[i] = sum over b < n of per_sample[b * per + i] in batch order (conv_grad_simt.cu; the stem data gradient of planes shared by
// the batch)
int stem_dgrad_batch_sum(const float* per_sample, float* out, int n, size_t per, cudaStream_t st);
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_grid_sync() {
  // wait only: the dependents are released when this grid's blocks exit (implicit trigger).  Releasing them at the top
  // (griddepcontrol.launch_dependents before the wait) measured 3% SLOWER on the sampler step and 8% on the training step:
  // blocks of the next kernels become resident early and take issue slots / shared memory from the running grid's tail.
  asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  if (pdl_enabled()) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  if (e != cudaSuccess) note_launch_error(e);
}
// the same launch as a thread-block cluster of `cluster_x` CTAs along x (gridDim.x must be a multiple of it)
template <typename... KArgs, typename... Args>
inline void launch_k_cluster(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, unsigned cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  attr[na].id = cudaLaunchAttributeClusterDimension;
  attr[na].val.clusterDim.x = cluster_x;
  attr[na].val.clusterDim.y = 1;
  attr[na].val.clusterDim.z = 1;
  ++na;
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
  if (e != cudaSuccess) note_launch_error(e);
}
#endif
inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

// ---- activation formats ---------------------------------------------------------------------
// A "vector" is 8 consecutive channels of one pixel.  Act<FMT>::load8 / store8 move one vector
// between global memory and fp32 registers.
template <int FMT>
struct Act;

template <>
struct Act<SBGM_FMT_F32> {
  static constexpr int kElemBytes = 4;
  __device__ __forceinline__ static void load8(const void* base, size_t, size_t idx, float (&v)[8]) {
    const float4* p = reinterpret_cast<const float4*>(static_cast<const float*>(base) + idx);
    float4 a = __ldg(p), b = __ldg(p + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  __device__ __forceinline__ static void store8(void* base, size_t, size_t idx, const float (&v)[8]) {
    float4* p = reinterpret_cast<float4*>(static_cast<float*>(base) + idx);
    p[0] = make_float4(v[0], v[1], v[2], v[3]);
    p[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
};

__device__ __forceinline__ void unpack_bf16x8(const uint4& u, float (&v)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ uint4 pack_bf16x8(const float (&v)[8]) {
  return make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
}
__device__ __forceinline__ float bf16_round(float a) { return __bfloat162float(__float2bfloat16_rn(a)); }

template <>
struct Act<SBGM_FMT_BF16> {
  static constexpr int kElemBytes = 2;
  __device__ __forceinline__ static void load8(const void* base, size_t, size_t idx, float (&v)[8]) {
    uint4 u = __ldg(reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(base) + idx));
    unpack_bf16x8(u, v);
  }
  __device__ __forceinline__ static void store8(void* base, size_t, size_t idx, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(static_cast<__nv_bfloat16*>(base) + idx) = pack_bf16x8(v);
  }
};

template <>
struct Act<SBGM_FMT_BF16X2> {
  static constexpr int kElemBytes = 2;
  __device__ __forceinline__ static void load8(const void* base, size_t plane, size_t idx, float (&v)[8]) {
    const __nv_bfloat16* p = static_cast<const __nv_bfloat16*>(base) + idx;
    uint4 uh = __ldg(reinterpret_cast<const uint4*>(p));
    uint4 ul = __ldg(reinterpret_cast<const uint4*>(p + plane));
    float lo[8];
    unpack_bf16x8(uh, v);
    unpack_bf16x8(ul, lo);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] += lo[i];
  }
  __device__ __forceinline__ static void store8(void* base, size_t plane, size_t idx, const float (&v)[8]) {
    __nv_bfloat16* p = static_cast<__nv_bfloat16*>(base) + idx;
    float hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      hi[i] = bf16_round(v[i]);
      lo[i] = v[i] - hi[i];
    }
    *reinterpret_cast<uint4*>(p) = pack_bf16x8(hi);
    *reinterpret_cast<uint4*>(p + plane) = pack_bf16x8(lo);
  }
};

// float16 plane.  Stores saturate to +-65504 (cvt.rn.satfinite): an activation outside the float16 range clamps instead of
// becoming inf -> NaN three layers later; everything behind a normalisation layer is O(10).
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %2, %1;" : "=r"(r) : "f"(a), "f"(b));     // low half = a
  return r;
}
__device__ __forceinline__ uint4 pack_f16x8(const float (&v)[8]) {
  return make_uint4(pack_f16x2(v[0], v[1]), pack_f16x2(v[2], v[3]), pack_f16x2(v[4], v[5]), pack_f16x2(v[6], v[7]));
}
__device__ __forceinline__ void unpack_f16x8(const uint4& u, float (&v)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
__device__ __forceinline__ float f16_round(float a) {
  const uint32_t p = pack_f16x2(a, 0.0f);
  return __half2float(__ushort_as_half(static_cast<unsigned short>(p & 0xffffu)));
}

template <>
struct Act<SBGM_FMT_F16> {
  static constexpr int kElemBytes = 2;
  __device__ __forceinline__ static void load8(const void* base, size_t, size_t idx, float (&v)[8]) {
    uint4 u = __ldg(reinterpret_cast<const uint4*>(static_cast<const __half*>(base) + idx));
    unpack_f16x8(u, v);
  }
  __device__ __forceinline__ static void store8(void* base, size_t, size_t idx, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(static_cast<__half*>(base) + idx) = pack_f16x8(v);
  }
};

// Storage traits of the tensor-core formats: activation planes, weight planes, element rounding / packing.
template <int FMT>
struct TcFmt {
  static constexpr int kAPlanes = (FMT == SBGM_FMT_BF16X2) ? 2 : 1;                        // activation planes
  static constexpr int kBPlanes = (FMT == SBGM_FMT_BF16X2 || FMT == SBGM_FMT_F16) ? 2 : 1;  // weight planes
  static constexpr bool kHalf = (FMT == SBGM_FMT_F16);                                     // float16 (else bfloat16) elements
  // factor of the second weight plane's product when the accumulator halves are summed
  static constexpr float kLoScale = kHalf ? (1.0f / SBGM_F16_WLO_SCALE) : 1.0f;
  __device__ __forceinline__ static float round(float x) { return kHalf ? f16_round(x) : bf16_round(x); }
  // two values through one pack instruction
  __device__ __forceinline__ static void round2(float& a, float& b) {
    if (kHalf) {
      const uint32_t p = pack_f16x2(a, b);
      a = __half2float(__ushort_as_half(static_cast<unsigned short>(p & 0xffffu)));
      b = __half2float(__ushort_as_half(static_cast<unsigned short>(p >> 16)));
    } else {
      const uint32_t p = pack_bf16x2(a, b);
      a = __uint_as_float(p << 16);
      b = __uint_as_float(p & 0xffff0000u);
    }
  }
  __device__ __forceinline__ static uint4 pack8(const float (&v)[8]) { return kHalf ? pack_f16x8(v) : pack_bf16x8(v); }
};

// Dispatch a templated launcher on the runtime format id.
#define SBGM_DISPATCH_FMT(fmt, ...)                                         \
  switch (fmt) {                                                             \
    case SBGM_FMT_F32: { constexpr int FMT = SBGM_FMT_F32; __VA_ARGS__; break; }       \
    case SBGM_FMT_BF16: { constexpr int FMT = SBGM_FMT_BF16; __VA_ARGS__; break; }     \
    case SBGM_FMT_BF16X2: { constexpr int FMT = SBGM_FMT_BF16X2; __VA_ARGS__; break; } \
    case SBGM_FMT_F16: { constexpr int FMT = SBGM_FMT_F16; __VA_ARGS__; break; }       \
    default: ::sbgm::set_error("unknown activation format %d", fmt); return 1;          \
  }

// ---- small math ---------------------------------------------------------------------------
// SiLU with the hardware exp2 / reciprocal (MUFU): ~2 ulp, against a 1e-3 parity gate; the GroupNorm+SiLU pass over the
// 64x64 maps was instruction-bound (not HBM-bound) with the IEEE expf + division sequence.
__device__ __forceinline__ float silu(float x) { return __fdividef(x, 1.0f + __expf(-x)); }
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float apply_act(float x, int act) {
  switch (act) {
    case SBGM_ACT_RELU: return fmaxf(x, 0.0f);
    case SBGM_ACT_SILU: return silu(x);
    case SBGM_ACT_GELU: return gelu_erf(x);
    default: return x;
  }
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- Philox4x32-10 (Salmon et al. 2011); stream layout documented in oracle/philox_ref.py ----
struct Philox {
  __device__ __forceinline__ static uint4 rand4(uint64_t q, uint32_t draw, uint64_t seed) {
    uint32_t c0 = static_cast<uint32_t>(q), c1 = static_cast<uint32_t>(q >> 32), c2 = draw, c3 = 0u;
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
      c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
  __device__ __forceinline__ static float u01(uint32_t r) {
    return (static_cast<float>(r >> 8) + 0.5f) * 5.9604644775390625e-08f;  // 2^-24
  }
  // four standard normals for elements 4q .. 4q+3
  __device__ __forceinline__ static float4 normal4(uint64_t q, uint32_t draw, uint64_t seed) {
    const uint4 r = rand4(q, draw, seed);
    float4 z;
    float s, c;
    const float rad0 = sqrtf(-2.0f * logf(u01(r.x)));
    sincosf(6.2831855f * u01(r.y), &s, &c);
    z.x = rad0 * c; z.y = rad0 * s;
    const float rad1 = sqrtf(-2.0f * logf(u01(r.z)));
    sincosf(6.2831855f * u01(r.w), &s, &c);
    z.z = rad1 * c; z.w = rad1 * s;
    return z;
  }
  __device__ __forceinline__ static float4 uniform4(uint64_t q, uint32_t draw, uint64_t seed) {
    const uint4 r = rand4(q, draw, seed);
    return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
  }
};

}  // namespace sbgm
