// attention_bwd.cu -- backward of the attention core softmax(Q K^T / sqrt(d)) V of ImageSelfAttention
// (sbgm/score_unet.py:112-148; torch autograd through nn.MultiheadAttention in the reference).
//
// The attention blocks sit on the 4x4 .. 16x16 maps (S <= 1024 tokens): ~3% of the network FLOPs.  The backward
// works head-major in fp32 from a workspace:
//   unpack qkv, dO -> Q, K, V, dO [b*heads][S][d];   P = softmax(scale Q K^T);   dP = dO V^T;
//   dS = P o (dP - rowsum(P o dP));   dV = P^T dO;   dQ = scale dS K;   dK = scale dS^T Q;   pack -> dqkv.
// The five products run through one batched CUDA-core GEMM (64x64x16 tiles, 4x4 per thread).
#include "common.cuh"

namespace sbgm {

template <int FMT>
__global__ void attn_unpack_kernel(const void* __restrict__ qkv, size_t qkv_plane, const void* __restrict__ dout, size_t dout_plane,
                                   float* __restrict__ q, float* __restrict__ k, float* __restrict__ v, float* __restrict__ go,
                                   int b, int s, int c, int heads) {
  pdl_grid_sync();
  const int d = c / heads, dvec = d >> 3, cvec = c >> 3;
  const uint32_t total = static_cast<uint32_t>(b) * s * cvec;          // 32-bit divisions only
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int vec = static_cast<int>(i % cvec);
    const uint32_t tok = i / cvec;
    const int head = vec / dvec, dv = vec - head * dvec;
    const size_t bi = tok / static_cast<uint32_t>(s), si = tok - bi * s;
    const size_t dst = ((bi * heads + head) * s + si) * d + dv * 8;
    float t[8];
    Act<FMT>::load8(qkv, qkv_plane, static_cast<size_t>(tok) * 3 * c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) q[dst + j] = t[j];
    Act<FMT>::load8(qkv, qkv_plane, static_cast<size_t>(tok) * 3 * c + c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) k[dst + j] = t[j];
    Act<FMT>::load8(qkv, qkv_plane, static_cast<size_t>(tok) * 3 * c + 2 * c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[dst + j] = t[j];
    Act<FMT>::load8(dout, dout_plane, static_cast<size_t>(tok) * c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) go[dst + j] = t[j];
  }
}

template <int FMT>
__global__ void attn_pack_kernel(const float* __restrict__ dq, const float* __restrict__ dk, const float* __restrict__ dv,
                                 void* __restrict__ dqkv, size_t plane, int b, int s, int c, int heads) {
  pdl_grid_sync();
  const int d = c / heads, dvec = d >> 3, cvec = c >> 3;
  const uint32_t total = static_cast<uint32_t>(b) * s * cvec;          // 32-bit divisions only
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int vec = static_cast<int>(i % cvec);
    const uint32_t tok = i / cvec;
    const int head = vec / dvec, dvi = vec - head * dvec;
    const size_t bi = tok / static_cast<uint32_t>(s), si = tok - bi * s;
    const size_t src = ((bi * heads + head) * s + si) * d + dvi * 8;
    float t[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = dq[src + j];
    Act<FMT>::store8(dqkv, plane, static_cast<size_t>(tok) * 3 * c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = dk[src + j];
    Act<FMT>::store8(dqkv, plane, static_cast<size_t>(tok) * 3 * c + c + vec * 8, t);
#pragma unroll
    for (int j = 0; j < 8; ++j) t[j] = dv[src + j];
    Act<FMT>::store8(dqkv, plane, static_cast<size_t>(tok) * 3 * c + 2 * c + vec * 8, t);
  }
}

// C[z][M][N] = alpha * op(A[z]) op(B[z]);  A is [M][K] (TA: [K][M]), B is [K][N] (TB: [N][K]); row-major, dense.
template <bool TA, bool TB>
__global__ void __launch_bounds__(256)
bgemm_kernel(const float* __restrict__ A, const float* __restrict__ B, float* __restrict__ C, int M, int N, int K, float alpha,
             size_t strideA, size_t strideB, size_t strideC) {
  pdl_grid_sync();
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const float* a = A + blockIdx.z * strideA;
  const float* bm = B + blockIdx.z * strideB;
  float* cm = C + blockIdx.z * strideC;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    __syncthreads();
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int item = threadIdx.x + e * 256;
      // A tile: element (mm, kk); choose the mapping that walks memory contiguously
      const int kk_a = TA ? item >> 6 : item & 15, mm = TA ? item & 63 : item >> 4;
      const int gm = m0 + mm, gk = k0 + kk_a;
      As[kk_a][mm] = (gm < M && gk < K) ? (TA ? a[static_cast<size_t>(gk) * M + gm] : a[static_cast<size_t>(gm) * K + gk]) : 0.0f;
      const int kk_b = TB ? item & 15 : item >> 6, nn = TB ? item >> 4 : item & 63;
      const int gn = n0 + nn, gkb = k0 + kk_b;
      Bs[kk_b][nn] = (gn < N && gkb < K) ? (TB ? bm[static_cast<size_t>(gn) * K + gkb] : bm[static_cast<size_t>(gkb) * N + gn]) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn < N) cm[static_cast<size_t>(gm) * N + gn] = alpha * acc[i][j];
    }
  }
}

// One warp per row: p <- softmax(p);  ds <- p o (ds - sum(p o ds))   (ds holds dP on entry)
__global__ void attn_softmax_bwd_kernel(float* __restrict__ p, float* __restrict__ ds, size_t rows, int s) {
  pdl_grid_sync();
  const size_t row = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* pr = p + row * s;
  float* dr = ds + row * s;
  float m = -INFINITY;
  for (int j = lane; j < s; j += 32) m = fmaxf(m, pr[j]);
  m = warp_max(m);
  float l = 0.0f;
  for (int j = lane; j < s; j += 32) {
    const float e = expf(pr[j] - m);
    pr[j] = e;
    l += e;
  }
  l = warp_sum(l);
  const float inv = 1.0f / l;
  float dsum = 0.0f;
  for (int j = lane; j < s; j += 32) {
    const float pv = pr[j] * inv;
    pr[j] = pv;
    dsum = fmaf(pv, dr[j], dsum);
  }
  dsum = warp_sum(dsum);
  for (int j = lane; j < s; j += 32) dr[j] = pr[j] * (dr[j] - dsum);
}

template <bool TA, bool TB>
static void launch_bgemm(const float* A, const float* B, float* C, int M, int N, int K, float alpha, size_t sA, size_t sB, size_t sC,
                         int batch, cudaStream_t st) {
  dim3 grid(ceil_div(N, 64), ceil_div(M, 64), batch);
  launch_k((bgemm_kernel<TA, TB>), grid, 256, 0, st, A, B, C, M, N, K, alpha, sA, sB, sC);
}

}  // namespace sbgm

namespace sbgm {
int attention_bwd_mma_dispatch(const void* qkv, const void* out, const void* dout, void* dqkv, int fmt, int b, int s, int c, int heads,
                               cudaStream_t st);     // attention_bwd_mma.cu; -1 = shape / format not covered
}

using namespace sbgm;

extern "C" {

size_t sbgm_attention_backward_scratch_floats(int b, int s, int c, int heads) {
  (void)heads;
  return static_cast<size_t>(7) * b * s * c + static_cast<size_t>(2) * b * heads * s * s;
}

int sbgm_attention_backward(const void* qkv, size_t qkv_plane, const void* out, size_t out_plane, const void* dout, size_t dout_plane,
                            void* dqkv, size_t dqkv_plane, int fmt, int b, int s, int c, int heads, float* scratch, void* stream) {
  SBGM_REQUIRE(heads >= 1 && c % heads == 0 && (c / heads) % 8 == 0, "attention_backward: bad c=%d heads=%d", c, heads);
  cudaStream_t st = as_stream(stream);
  (void)out_plane;
  // bf16, S % 16 == 0, head dim 32 / 64 / 128: one tensor-core launch
  const int mma_rc = attention_bwd_mma_dispatch(qkv, out, dout, dqkv, fmt, b, s, c, heads, st);
  if (mma_rc >= 0) return mma_rc;
  const int d = c / heads, bh = b * heads;
  const size_t tok = static_cast<size_t>(b) * s * c, mat = static_cast<size_t>(bh) * s * s;
  float* q = scratch;
  float* k = q + tok;
  float* v = k + tok;
  float* go = v + tok;
  float* dq = go + tok;
  float* dk = dq + tok;
  float* dv = dk + tok;
  float* p = dv + tok;
  float* ds = p + mat;
  const float scale = 1.0f / sqrtf(static_cast<float>(d));
  const size_t items = static_cast<size_t>(b) * s * (c / 8);
  const int g = static_cast<int>(items / 256 + 1 < 148 * 8 ? items / 256 + 1 : 148 * 8);
  SBGM_DISPATCH_FMT(fmt, (launch_k((attn_unpack_kernel<FMT>), g, 256, 0, st, qkv, qkv_plane, dout, dout_plane, q, k, v, go, b, s, c, heads)));
  const size_t sd = static_cast<size_t>(s) * d, ss = static_cast<size_t>(s) * s;
  launch_bgemm<false, true>(q, k, p, s, s, d, scale, sd, sd, ss, bh, st);        // S = scale Q K^T
  launch_bgemm<false, true>(go, v, ds, s, s, d, 1.0f, sd, sd, ss, bh, st);       // dP = dO V^T
  const size_t rows = static_cast<size_t>(bh) * s;
  launch_k((attn_softmax_bwd_kernel), ceil_div(static_cast<long long>(rows) * 32, 256), 256, 0, st, p, ds, rows, s);
  launch_bgemm<true, false>(p, go, dv, s, d, s, 1.0f, ss, sd, sd, bh, st);       // dV = P^T dO
  launch_bgemm<false, false>(ds, k, dq, s, d, s, scale, ss, sd, sd, bh, st);     // dQ = scale dS K
  launch_bgemm<true, false>(ds, q, dk, s, d, s, scale, ss, sd, sd, bh, st);      // dK = scale dS^T Q
  SBGM_DISPATCH_FMT(fmt, (launch_k((attn_pack_kernel<FMT>), g, 256, 0, st, dq, dk, dv, dqkv, dqkv_plane, b, s, c, heads)));
  return check_launch("attention_backward");
}

}  // extern "C"
