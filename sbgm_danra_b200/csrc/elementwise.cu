// elementwise.cu -- bandwidth-bound kernels of the score-UNet: layout conversion, time embedding
// + projections, GroupNorm(+skip+time+activation), LayerNorm, bilinear x2 upsample and the
// final cout<=4 convolution fused with the 1/std scaling.  All are coalesced over the NHWC
// channel axis with 8-channel (16 or 32 byte) vectors per thread.
#include <stdarg.h>

#include "common.cuh"
#include <mutex>
#include <unordered_map>

namespace sbgm {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
static thread_local cudaError_t g_launch_err = cudaSuccess;
void note_launch_error(cudaError_t e) { g_launch_err = e; }
bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("SBGM_B200_PDL");
    v = (e != nullptr && e[0] == '0') ? 0 : 1;
  }
  return v != 0;
}
int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess && g_launch_err != cudaSuccess) e = g_launch_err;
  g_launch_err = cudaSuccess;
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return 2;
  }
  return 0;
}

// ---- layout conversion ----------------------------------------------------------------------
// NCHW fp32 -> NHWC fmt via a 32(pixels) x 8k(channels) smem transpose.
template <int FMT>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ src, void* __restrict__ dst, size_t plane, int c, int hw) {
  pdl_grid_sync();
  // block: 32 pixels x 64 channels tile; grid (hw/32, c/64 (ceil), n)
  __shared__ float tile[64][33];
  const int n = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 256 threads: 32 x 8
  for (int cc = ty; cc < 64; cc += 8) {
    const int ch = c0 + cc, p = p0 + tx;
    tile[cc][tx] = (ch < c && p < hw) ? __ldg(src + (static_cast<size_t>(n) * c + ch) * hw + p) : 0.0f;
  }
  __syncthreads();
  // each thread writes one 8-channel vector: 32 pixels x 8 vectors = 256
  const int pix = threadIdx.x >> 3, vec = threadIdx.x & 7;
  const int p = p0 + pix, ch = c0 + vec * 8;
  if (p < hw && ch < c) {
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = tile[vec * 8 + i][pix];
    Act<FMT>::store8(dst, plane, (static_cast<size_t>(n) * hw + p) * c + ch, v);
  }
}

template <int FMT>
__global__ void nhwc_to_nchw_kernel(const void* __restrict__ src, size_t plane, float* __restrict__ dst, int c, int hw) {
  pdl_grid_sync();
  __shared__ float tile[64][33];
  const int n = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 32;
  const int pix = threadIdx.x >> 3, vec = threadIdx.x & 7;
  {
    const int p = p0 + pix, ch = c0 + vec * 8;
    float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (p < hw && ch < c) Act<FMT>::load8(src, plane, (static_cast<size_t>(n) * hw + p) * c + ch, v);
#pragma unroll
    for (int i = 0; i < 8; ++i) tile[vec * 8 + i][pix] = v[i];
  }
  __syncthreads();
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int cc = ty; cc < 64; cc += 8) {
    const int ch = c0 + cc, p = p0 + tx;
    if (ch < c && p < hw) dst[(static_cast<size_t>(n) * c + ch) * hw + p] = tile[cc][tx];
  }
}

template <int SRC, int DST>
__global__ void convert_kernel(const void* __restrict__ src, size_t sp, void* __restrict__ dst, size_t dp, size_t nvec) {
  pdl_grid_sync();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < nvec;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float v[8];
    Act<SRC>::load8(src, sp, i * 8, v);
    Act<DST>::store8(dst, dp, i * 8, v);
  }
}

// ---- time embedding + projections -----------------------------------------------------------
// One block per row (batch member or sampler step).  Phase 1: the n_sets Gaussian-Fourier
// embeddings (+ label embedding on set 0), SiLU applied, into shared memory.  Phase 2: one warp
// per output channel does the te-long dot product.
constexpr int kTimeProjCols = 128;   // output channels per block
__global__ void time_embed_project_kernel(const float* __restrict__ t, int t_row_stride, int t_step_stride,
                                          const int32_t* __restrict__ step_counter, const int64_t* __restrict__ y,
                                          const float* __restrict__ fw, int n_sets, int te,
                                          const float* __restrict__ label_emb, const float* __restrict__ pw,
                                          const float* __restrict__ pb, const int32_t* __restrict__ pset,
                                          int c_total, float* __restrict__ out) {
  pdl_grid_sync();
  extern __shared__ float emb[];  // [n_sets][te], SiLU already applied
  const int row = blockIdx.x, half = te / 2;
  const int step = step_counter ? *step_counter : 0;
  const float tv = t[static_cast<size_t>(row) * t_row_stride + static_cast<size_t>(step) * t_step_stride];
  const int64_t lab = (y != nullptr) ? y[row] : -1;
  for (int i = threadIdx.x; i < n_sets * half; i += blockDim.x) {
    const int s = i / half, j = i - s * half;
    // same association order as the reference: (t * W) * 2pi  (score_unet.py:44)
    const float arg = (tv * fw[i]) * 6.283185307179586f;
    float sv, cv;
    sincosf(arg, &sv, &cv);
    if (s == 0 && lab >= 0 && label_emb != nullptr) {
      sv += label_emb[lab * te + j];
      cv += label_emb[lab * te + half + j];
    }
    emb[s * te + j] = silu(sv);
    emb[s * te + half + j] = silu(cv);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
  const int c_begin = blockIdx.y * kTimeProjCols, c_end = min(c_total, c_begin + kTimeProjCols);
  for (int c = c_begin + warp; c < c_end; c += nwarp) {
    const float* e = emb + pset[c] * te;
    const float* wrow = pw + static_cast<size_t>(c) * te;
    float acc = 0.0f;
    for (int k = lane; k < te; k += 32) acc = fmaf(e[k], __ldg(wrow + k), acc);
    acc = warp_sum(acc);
    if (lane == 0) out[static_cast<size_t>(row) * c_total + c] = acc + pb[c];
  }
}

__global__ void fourier_embed_kernel(const float* __restrict__ t, const float* __restrict__ fw, int half,
                                     float* __restrict__ out, int rows) {
  pdl_grid_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * half) return;
  const int row = i / half, j = i - row * half;
  float sv, cv;
  sincosf((t[row] * fw[j]) * 6.283185307179586f, &sv, &cv);
  out[static_cast<size_t>(row) * 2 * half + j] = sv;
  out[static_cast<size_t>(row) * 2 * half + half + j] = cv;
}

__global__ void cfg_combine_kernel(const float* __restrict__ sc, const float* __restrict__ su, float scale,
                                   float* __restrict__ out, size_t count) {
  pdl_grid_sync();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < count;
       i += static_cast<size_t>(gridDim.x) * blockDim.x)
    out[i] = (1.0f + scale) * sc[i] - scale * su[i];
}

__global__ void select_step_row_kernel(const float* __restrict__ table, int cols, const int32_t* __restrict__ step,
                                       float* __restrict__ out) {
  pdl_grid_sync();
  const float* row = table + static_cast<size_t>(*step) * cols;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < cols; i += gridDim.x * blockDim.x) out[i] = row[i];
}

// ---- GroupNorm ------------------------------------------------------------------------------
// Stage 1: per (n, chunk) partial per-GROUP sum / sum-of-squares (deterministic, no atomics).
// Block = 256 threads = (c/8 channel vectors) x (256/(c/8) pixel lanes); c in {64..512}.
constexpr int kGnChunks = 32;

template <int FMT>
__global__ void gn_partial_kernel(const void* __restrict__ x, size_t plane, int hw, int c, int groups,
                                  float* __restrict__ partials, int chunks) {
  pdl_grid_sync();
  extern __shared__ float red[];  // [lanes][c][2] then [c][2]
  const int n = blockIdx.y, chunk = blockIdx.x;
  const int vecs = c >> 3, lanes = blockDim.x / vecs;
  const int vec = threadIdx.x % vecs, lane = threadIdx.x / vecs;
  const int per_chunk = (hw + chunks - 1) / chunks;
  const int p_begin = chunk * per_chunk, p_end = min(hw, p_begin + per_chunk);
  float s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, q[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (lane < lanes) {
    for (int p = p_begin + lane; p < p_end; p += lanes) {
      float v[8];
      Act<FMT>::load8(x, plane, (static_cast<size_t>(n) * hw + p) * c + vec * 8, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] += v[i];
        q[i] = fmaf(v[i], v[i], q[i]);
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      red[(lane * c + vec * 8 + i) * 2] = s[i];
      red[(lane * c + vec * 8 + i) * 2 + 1] = q[i];
    }
  }
  __syncthreads();
  float* chan = red + static_cast<size_t>(lanes) * c * 2;  // [c][2]
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    float ss = 0.0f, qq = 0.0f;
    for (int l = 0; l < lanes; ++l) {
      ss += red[(l * c + ch) * 2];
      qq += red[(l * c + ch) * 2 + 1];
    }
    chan[2 * ch] = ss;
    chan[2 * ch + 1] = qq;
  }
  __syncthreads();
  const int cpg = c / groups;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {
    float ss = 0.0f, qq = 0.0f;
    for (int j = 0; j < cpg; ++j) {
      ss += chan[2 * (g * cpg + j)];
      qq += chan[2 * (g * cpg + j) + 1];
    }
    float* o = partials + ((static_cast<size_t>(n) * chunks + chunk) * groups + g) * 2;
    o[0] = ss;
    o[1] = qq;
  }
}

// Stage 2: finish the reduction per group (double accumulation over the 32 chunks) and apply.
template <int FMT>
__global__ void gn_apply_kernel(const void* __restrict__ x, size_t x_plane, const float* __restrict__ partials,
                                int chunks, int pgroups, const float* __restrict__ gamma, const float* __restrict__ beta, int groups, float eps,
                                const void* __restrict__ skip, size_t skip_plane, const float* __restrict__ tproj,
                                int tproj_stride, int act, void* __restrict__ y, size_t y_plane, int hw, int c) {
  pdl_grid_sync();
  extern __shared__ float coef[];  // [c][2]: scale, shift per channel (norm + affine + tproj folded), then [groups][2]
  float* gstat = coef + 2 * c;
  const int n = blockIdx.y;
  const int cpg = c / groups;
  // finish the reduction over chunks: one warp per group (lanes stride the chunks, double accumulation, fixed order)
  {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarp = blockDim.x >> 5;
    for (int g = warp; g < groups; g += nwarp) {
      double s = 0.0, q = 0.0;
      const int sub = pgroups / groups;      // partial groups per group (1 for the stand-alone statistics kernel)
      for (int k = lane; k < chunks * sub; k += 32) {
        const int ck = k / sub, sg = k - ck * sub;
        const float2 p = __ldg(reinterpret_cast<const float2*>(partials + ((static_cast<size_t>(n) * chunks + ck) * pgroups + g * sub + sg) * 2));
        s += p.x;
        q += p.y;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        q += __shfl_xor_sync(0xffffffffu, q, o);
      }
      if (lane == 0) {
        const double cnt = static_cast<double>(hw) * cpg;
        const double mean = s / cnt;
        const double var = fmax(q / cnt - mean * mean, 0.0);
        gstat[2 * g] = static_cast<float>(mean);
        gstat[2 * g + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
      }
    }
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < c; ch += blockDim.x) {
    const int g = ch / cpg;
    const float ga = gamma ? gamma[ch] : 1.0f, be = beta ? beta[ch] : 0.0f;
    const float sc = gstat[2 * g + 1] * ga;
    float sh = be - gstat[2 * g] * sc;
    if (tproj) sh += tproj[static_cast<size_t>(n) * tproj_stride + ch];
    coef[2 * ch] = sc;
    coef[2 * ch + 1] = sh;
  }
  __syncthreads();
  const int vecs = c >> 3;
  const uint32_t total = static_cast<uint32_t>(hw) * vecs;          // < 2^32 (host-checked)
  const uint32_t stride = gridDim.x * blockDim.x;
  const int vec = static_cast<int>((blockIdx.x * blockDim.x + threadIdx.x) % vecs);
  float sc8[8], sh8[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sc8[j] = coef[2 * (vec * 8 + j)];
    sh8[j] = coef[2 * (vec * 8 + j) + 1];
  }
  const bool fixed_vec = (stride % vecs) == 0;                      // always for power-of-two channel counts
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    if (!fixed_vec) {
      const int vv = static_cast<int>(i % vecs);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        sc8[j] = coef[2 * (vv * 8 + j)];
        sh8[j] = coef[2 * (vv * 8 + j) + 1];
      }
    }
    const size_t idx = (static_cast<size_t>(n) * hw) * c + static_cast<size_t>(i) * 8;
    float v[8];
    Act<FMT>::load8(x, x_plane, idx, v);
    if (skip) {
      float sk[8];
      Act<FMT>::load8(skip, skip_plane, idx, sk);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc8[j], sh8[j]) + sk[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = fmaf(v[j], sc8[j], sh8[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = apply_act(v[j], act);
    Act<FMT>::store8(y, y_plane, idx, v);
  }
}

// ---- LayerNorm: one warp per token row --------------------------------------------------------
template <int FMT>
__global__ void layernorm_kernel(const void* __restrict__ x, size_t x_plane, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, float eps, void* __restrict__ y, size_t y_plane,
                                 int rows, int c) {
  pdl_grid_sync();
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int vecs = c >> 3;  // <= 64 -> at most 2 vectors per lane
  float v[2][8];
  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int vec = lane + 32 * k;
    if (vec < vecs) {
      Act<FMT>::load8(x, x_plane, static_cast<size_t>(row) * c + vec * 8, v[k]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[k][j];
    }
  }
  const float mean = warp_sum(s) / c;
  float q = 0.0f;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    if (lane + 32 * k < vecs) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[k][j] - mean;
        q = fmaf(d, d, q);
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / c + eps);
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int vec = lane + 32 * k;
    if (vec < vecs) {
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[k][j] - mean) * rstd * gamma[vec * 8 + j] + beta[vec * 8 + j];
      Act<FMT>::store8(y, y_plane, static_cast<size_t>(row) * c + vec * 8, o);
    }
  }
}

// ---- bilinear x2 upsample, align_corners=False ------------------------------------------------
// One thread per (input pixel, 8-channel vector): the 3x3 clamped neighbourhood (9 vector loads) yields the
// 2x2 output block.  ATen's rule src = max(0, (dst + 0.5) / 2 - 0.5) gives, for output row 2i: rows (i-1, i)
// with weights (0.25, 0.75) [row 0: (0,0) -> in[0]]; for row 2i+1: rows (i, min(i+1, h-1)) with (0.75, 0.25).
template <int FMT>
__global__ void upsample2x_kernel(const void* __restrict__ x, size_t x_plane, void* __restrict__ y, size_t y_plane,
                                  int n, int h, int w, int c) {
  pdl_grid_sync();
  const uint32_t vecs = c >> 3;
  const uint32_t total = static_cast<uint32_t>(n) * h * w * vecs;   // < 2^32 (host-checked): 32-bit divisions only
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int vec = static_cast<int>(i % vecs);
    uint32_t r = i / vecs;
    const int ix = static_cast<int>(r % w);
    r /= w;
    const int iy = static_cast<int>(r % h);
    const int b = static_cast<int>(r / h);
    const int ys[3] = {max(iy - 1, 0), iy, min(iy + 1, h - 1)};
    const int xs[3] = {max(ix - 1, 0), ix, min(ix + 1, w - 1)};
    float v[3][3][8];
    const size_t base = static_cast<size_t>(b) * h * w;
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int e = 0; e < 3; ++e)
        Act<FMT>::load8(x, x_plane, (base + static_cast<size_t>(ys[a]) * w + xs[e]) * c + vec * 8, v[a][e]);
    // ATen evaluates  h0 * (w0 * p00 + w1 * p01) + h1 * (w0 * p10 + w1 * p11)  with h1 = lambda, h0 = 1 - lambda
    const float l0 = (iy == 0) ? 0.0f : 0.75f, m0 = (ix == 0) ? 0.0f : 0.75f;   // lambda of the even output row / col
#pragma unroll
    for (int py = 0; py < 2; ++py) {
      constexpr int kDummy = 0; (void)kDummy;
      const int ra = py, rb = py + 1;        // static tap rows in v[][] (the clamped loads make borders exact)
      const float ly = (py == 0) ? l0 : 0.25f, hy = 1.0f - ly;
#pragma unroll
      for (int px = 0; px < 2; ++px) {
        const int ca = px, cb = px + 1;
        const float lx = (px == 0) ? m0 : 0.25f, hx = 1.0f - lx;
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          o[j] = hy * (hx * v[ra][ca][j] + lx * v[ra][cb][j]) + ly * (hx * v[rb][ca][j] + lx * v[rb][cb][j]);
        const size_t opix = (static_cast<size_t>(b) * 2 * h + 2 * iy + py) * 2 * w + 2 * ix + px;
        Act<FMT>::store8(y, y_plane, opix * c + vec * 8, o);
      }
    }
  }
}

// ---- stem im2col -------------------------------------------------------------------------------------------
// A block owns 32 output pixels of one output row and one input channel: the 8 x 70 input window goes through shared
// memory (coalesced row reads; every input value is used by 16 taps), then thread (pixel, window row r) writes that
// row's 8 taps as one vector -- 8 consecutive threads fill one 128-byte line.  (The direct form, 8 scalar loads per
// thread at 32 distinct lines per warp instruction, ran at the LSU wavefront limit: 374 us for the 7-channel C4 stem.)
template <int FMT>
__global__ void __launch_bounds__(256)
stem_im2col_kernel(const float* __restrict__ x, const float* __restrict__ planes, int np, int cc, int c_begin, int nch,
                   void* __restrict__ out, size_t out_plane, int n, int h, int w) {
  pdl_grid_sync();
  __shared__ float tile[8][72];
  const int ho = h / 2, wo = w / 2;
  const int ox0 = blockIdx.x * 32, oy = blockIdx.y;
  const int b = blockIdx.z / nch, cl = blockIdx.z - b * nch;
  const int c = c_begin + cl;
  const float* src = (c == 0) ? x + static_cast<size_t>(b) * h * w
                              : planes + (static_cast<size_t>(np == 1 ? 0 : b) * cc + (c - 1)) * h * w;
  for (int i = threadIdx.x; i < 8 * 70; i += 256) {
    const int r = i / 70, col = i - r * 70;
    const int iy = 2 * oy + r - 3, ix = 2 * ox0 + col - 3;
    tile[r][col] = (iy >= 0 && iy < h && ix >= 0 && ix < w) ? __ldg(src + static_cast<size_t>(iy) * w + ix) : 0.0f;
  }
  __syncthreads();
  const int r = threadIdx.x & 7, px = threadIdx.x >> 3;
  if (ox0 + px >= wo) return;
  float v[8];
#pragma unroll
  for (int s = 0; s < 8; ++s) v[s] = tile[r][2 * px + s];
  const size_t pix = (static_cast<size_t>(b) * ho + oy) * wo + ox0 + px;
  Act<FMT>::store8(out, out_plane, (pix * nch + cl) * 64 + r * 8, v);
}

// ---- final convolution: 3x3, cout <= 4, fused 1/std ---------------------------------------------
// One warp per output pixel: lanes split the 9*cin products (8 channels per lane per tap),
// warp-reduce, lane 0 writes.  Pure bandwidth: reads each input vector 9 times through L1/L2.
template <int FMT, int COUT>
__global__ void final_conv_kernel(const void* __restrict__ in, size_t plane, const float* __restrict__ wgt,
                                  const float* __restrict__ bias, const float* __restrict__ inv_std, int inv_stride,
                                  int inv_step_stride, const int32_t* __restrict__ step_counter,
                                  float* __restrict__ out, int n, int h, int w, int cin) {
  pdl_grid_sync();
  extern __shared__ float ws[];  // [COUT][9][cin]
  for (int i = threadIdx.x; i < COUT * 9 * cin; i += blockDim.x) ws[i] = wgt[i];
  __syncthreads();
  const int vecs = cin >> 3;
  const int lane = threadIdx.x & 31;
  const size_t npix = static_cast<size_t>(n) * h * w;
  const size_t warps_total = (static_cast<size_t>(gridDim.x) * blockDim.x) >> 5;
  for (size_t pix = (blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x) >> 5; pix < npix; pix += warps_total) {
    const int ox = static_cast<int>(pix % w);
    const int oy = static_cast<int>((pix / w) % h);
    const int b = static_cast<int>(pix / (static_cast<size_t>(w) * h));
    float acc[COUT];
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc[co] = 0.0f;
    for (int item = lane; item < 9 * vecs; item += 32) {
      const int tap = item / vecs, vec = item - tap * vecs;
      const int iy = oy + tap / 3 - 1, ix = ox + tap % 3 - 1;
      if (iy < 0 || iy >= h || ix < 0 || ix >= w) continue;
      float v[8];
      Act<FMT>::load8(in, plane, ((static_cast<size_t>(b) * h + iy) * w + ix) * cin + vec * 8, v);
#pragma unroll
      for (int co = 0; co < COUT; ++co) {
        const float* wp = ws + (co * 9 + tap) * cin + vec * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[co] = fmaf(v[j], wp[j], acc[co]);
      }
    }
#pragma unroll
    for (int co = 0; co < COUT; ++co) acc[co] = warp_sum(acc[co]);
    if (lane == 0) {
      const int step = step_counter ? *step_counter : 0;
      const float sc = inv_std ? inv_std[static_cast<size_t>(b) * inv_stride + static_cast<size_t>(step) * inv_step_stride] : 1.0f;
#pragma unroll
      for (int co = 0; co < COUT; ++co)
        out[((static_cast<size_t>(b) * COUT + co) * h + oy) * w + ox] = (acc[co] + bias[co]) * sc;
    }
  }
}

// out = (sum of the 9 per-tap partial products of the neighbours + bias) * scale; 4 pixels (one float4) per thread.
__global__ void final_gather_kernel(const float* __restrict__ proj, const float* __restrict__ bias,
                                    const float* __restrict__ inv_std, int inv_stride, int inv_step_stride,
                                    const int32_t* __restrict__ step_counter, float* __restrict__ out, int n, int h, int w) {
  pdl_grid_sync();
  const uint32_t total = static_cast<uint32_t>(n) * h * w;
  const int step = step_counter ? *step_counter : 0;
  const float b0 = bias[0];
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int x = static_cast<int>(i % w);
    const int y = static_cast<int>((i / w) % h);
    const int b = static_cast<int>(i / (static_cast<uint32_t>(w) * h));
    float acc = b0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int yy = y + r - 1;
      if (yy < 0 || yy >= h) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int xx = x + s - 1;
        if (xx < 0 || xx >= w) continue;
        acc += __ldg(proj + ((static_cast<size_t>(b) * h + yy) * w + xx) * SBGM_PROJ_STRIDE + r * 3 + s);
      }
    }
    const float sc = inv_std ? inv_std[static_cast<size_t>(b) * inv_stride + static_cast<size_t>(step) * inv_step_stride] : 1.0f;
    out[i] = acc * sc;
  }
}

// Blocks of `kern` that are resident at once on the whole GPU.  The GroupNorm apply pass (grid-stride, 48 registers: five
// blocks per SM) gets at most that many blocks: the fixed cap of 148 x 8 was 1.6 waves, i.e. it paid for two.
// (The same change left the bilinear upsample, 72 registers, unchanged to slightly slower: not applied there.)
int resident_blocks(const void* kern, int block, size_t smem) {
  static std::unordered_map<const void*, int> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(kern);
  if (it != cache.end()) return it->second;
  int per_sm = 0, dev = 0, sms = 148;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, block, smem) != cudaSuccess || per_sm < 1) per_sm = 4;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int v = per_sm * sms;
  cache[kern] = v;
  return v;
}

static int grid_for(size_t items, int block, int max_blocks = 148 * 16) {
  size_t g = (items + block - 1) / block;
  if (g < 1) g = 1;
  if (g > static_cast<size_t>(max_blocks)) g = max_blocks;
  return static_cast<int>(g);
}

}  // namespace sbgm

using namespace sbgm;

extern "C" {

const char* sbgm_last_error(void) { return g_err; }
int sbgm_version(void) { return 100; }
int sbgm_device_is_sm100(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10;
}

int sbgm_nchw_to_nhwc(const float* src, void* dst, size_t dst_plane, int fmt, int n, int c, int h, int w, void* stream) {
  SBGM_REQUIRE(c % 8 == 0, "nchw_to_nhwc: c=%d must be a multiple of 8", c);
  dim3 grid(ceil_div(h * w, 32), ceil_div(c, 64), n);
  SBGM_DISPATCH_FMT(fmt, (launch_k((nchw_to_nhwc_kernel<FMT>), grid, 256, 0, as_stream(stream), src, dst, dst_plane, c, h * w)));
  return check_launch("nchw_to_nhwc");
}
int sbgm_nhwc_to_nchw(const void* src, size_t src_plane, int fmt, float* dst, int n, int c, int h, int w, void* stream) {
  SBGM_REQUIRE(c % 8 == 0, "nhwc_to_nchw: c=%d must be a multiple of 8", c);
  dim3 grid(ceil_div(h * w, 32), ceil_div(c, 64), n);
  SBGM_DISPATCH_FMT(fmt, (launch_k((nhwc_to_nchw_kernel<FMT>), grid, 256, 0, as_stream(stream), src, src_plane, dst, c, h * w)));
  return check_launch("nhwc_to_nchw");
}

int sbgm_convert(const void* src, size_t sp, int sf, void* dst, size_t dp, int df, size_t count, void* stream) {
  SBGM_REQUIRE(count % 8 == 0, "convert: count must be a multiple of 8");
  const size_t nvec = count / 8;
  const int grid = grid_for(nvec, 256);
  cudaStream_t st = as_stream(stream);
#define SBGM_CVT(S, D) launch_k((convert_kernel<S, D>), grid, 256, 0, st, src, sp, dst, dp, nvec)
  if (sf == SBGM_FMT_F32 && df == SBGM_FMT_F32) SBGM_CVT(SBGM_FMT_F32, SBGM_FMT_F32);
  else if (sf == SBGM_FMT_F32 && df == SBGM_FMT_BF16) SBGM_CVT(SBGM_FMT_F32, SBGM_FMT_BF16);
  else if (sf == SBGM_FMT_F32 && df == SBGM_FMT_BF16X2) SBGM_CVT(SBGM_FMT_F32, SBGM_FMT_BF16X2);
  else if (sf == SBGM_FMT_BF16 && df == SBGM_FMT_F32) SBGM_CVT(SBGM_FMT_BF16, SBGM_FMT_F32);
  else if (sf == SBGM_FMT_BF16X2 && df == SBGM_FMT_F32) SBGM_CVT(SBGM_FMT_BF16X2, SBGM_FMT_F32);
  else if (sf == SBGM_FMT_F32 && df == SBGM_FMT_F16) SBGM_CVT(SBGM_FMT_F32, SBGM_FMT_F16);
  else if (sf == SBGM_FMT_F16 && df == SBGM_FMT_F32) SBGM_CVT(SBGM_FMT_F16, SBGM_FMT_F32);
  else { set_error("convert: unsupported format pair %d -> %d", sf, df); return 1; }
#undef SBGM_CVT
  return check_launch("convert");
}

int sbgm_time_embed_project(const float* t, int t_row_stride, int t_step_stride, const int32_t* step_counter,
                            const int64_t* y, const float* fourier_w, int n_sets, int te,
                            const float* label_emb, const float* proj_w, const float* proj_b,
                            const int32_t* proj_set, int c_total, float* out, int rows, void* stream) {
  SBGM_REQUIRE(te % 2 == 0 && n_sets >= 1 && rows >= 1, "time_embed_project: bad sizes te=%d sets=%d rows=%d", te, n_sets, rows);
  const size_t smem = static_cast<size_t>(n_sets) * te * sizeof(float);
  SBGM_REQUIRE(smem <= 48 * 1024, "time_embed_project: n_sets*te too large");
  launch_k((time_embed_project_kernel), dim3(rows, ceil_div(c_total, kTimeProjCols)), 256, smem, as_stream(stream), t, t_row_stride, t_step_stride, step_counter, y,
                                                                    fourier_w, n_sets, te, label_emb, proj_w, proj_b,
                                                                    proj_set, c_total, out);
  return check_launch("time_embed_project");
}

int sbgm_fourier_embed(const float* t, const float* fourier_w, int half, float* out, int rows, void* stream) {
  launch_k((fourier_embed_kernel), ceil_div(static_cast<long long>(rows) * half, 256), 256, 0, as_stream(stream), t, fourier_w, half, out, rows);
  return check_launch("fourier_embed");
}

int sbgm_cfg_combine(const float* s_cond, const float* s_uncond, float scale, float* out, size_t count, void* stream) {
  launch_k((cfg_combine_kernel), grid_for(count, 256), 256, 0, as_stream(stream), s_cond, s_uncond, scale, out, count);
  return check_launch("cfg_combine");
}

int sbgm_select_step_row(const float* table, int cols, const int32_t* step_counter, float* out, void* stream) {
  launch_k((select_step_row_kernel), ceil_div(cols, 256), 256, 0, as_stream(stream), table, cols, step_counter, out);
  return check_launch("select_step_row");
}

size_t sbgm_groupnorm_scratch_floats(int n, int c, int) { return static_cast<size_t>(n) * kGnChunks * c * 2; }  // upper bound (groups <= c)

int sbgm_groupnorm(const void* x, size_t x_plane, const float* gamma, const float* beta, int groups, float eps,
                   const void* skip, size_t skip_plane, const float* tproj, int tproj_stride, int act,
                   void* y, size_t y_plane, int fmt, int n, int hw, int c, float* partials, void* stream) {
  SBGM_REQUIRE(c % 8 == 0 && c <= 2048 && groups >= 1 && c % groups == 0, "groupnorm: bad c=%d groups=%d", c, groups);
  const int vecs = c / 8;
  SBGM_REQUIRE(vecs <= 256, "groupnorm: c too large");
  cudaStream_t st = as_stream(stream);
  const int lanes = 256 / vecs;
  const size_t smem1 = (static_cast<size_t>(lanes) + 1) * c * 2 * sizeof(float);
  const size_t smem2 = (static_cast<size_t>(c) + groups) * 2 * sizeof(float);
  // ~8 pixels per thread, at most kGnChunks chunks: the 8 x 8 x 512 map of the first decoder block was 32 chunks of TWO pixels
  // (2 048 blocks that mostly synchronise: 13.7 us for 4 MB)
  const int chunks = sbgm_norm_partials_chunks(hw, c);
  dim3 g1(chunks, n);
  int slots = 148 * 8;
  SBGM_DISPATCH_FMT(fmt, (slots = resident_blocks(reinterpret_cast<const void*>(gn_apply_kernel<FMT>), 256, smem2)));
  const int per_n_blocks = max(1, min(ceil_div(static_cast<long long>(hw) * vecs, 256 * 4), slots / max(n, 1)));
  dim3 g2(per_n_blocks, n);
  SBGM_DISPATCH_FMT(fmt, {
    launch_k((gn_partial_kernel<FMT>), g1, 256, smem1, st, x, x_plane, hw, c, groups, partials, chunks);
    launch_k((gn_apply_kernel<FMT>), g2, 256, smem2, st, x, x_plane, partials, chunks, groups, gamma, beta, groups, eps, skip,
                                                  skip_plane, tproj, tproj_stride, act, y, y_plane, hw, c);
  });
  return check_launch("groupnorm");
}

// Stage 1 alone: per (n, chunk) partial sums [n][32][groups][2]; groups == c gives the per-channel partials
// of train-mode BatchNorm (finished by sbgm_bn_stats_finalize / sbgm_gn_stats_finalize, backward.cu).
// chunk count of sbgm_norm_partials: ~8 pixels per thread, at most 32 (small maps get few chunks, so the finalize
// kernels sum few partials)
int sbgm_norm_partials_chunks(int hw, int c) {
  const int vecs = c / 8 > 0 ? c / 8 : 1;
  const int lanes = 256 / vecs > 0 ? 256 / vecs : 1;
  const int ch = hw / (lanes * 8);
  return ch < 1 ? 1 : (ch > kGnChunks ? kGnChunks : ch);
}

int sbgm_norm_partials(const void* x, size_t x_plane, int fmt, int n, int hw, int c, int groups, float* partials, void* stream) {
  SBGM_REQUIRE(c % 8 == 0 && c <= 2048 && groups >= 1 && c % groups == 0, "norm_partials: bad c=%d groups=%d", c, groups);
  const int vecs = c / 8;
  SBGM_REQUIRE(vecs <= 256, "norm_partials: c too large");
  const int lanes = 256 / vecs;
  const size_t smem1 = (static_cast<size_t>(lanes) + 1) * c * 2 * sizeof(float);
  const int chunks = sbgm_norm_partials_chunks(hw, c);
  dim3 g1(chunks, n);
  SBGM_DISPATCH_FMT(fmt, (launch_k((gn_partial_kernel<FMT>), g1, 256, smem1, as_stream(stream), x, x_plane, hw, c, groups, partials, chunks)));
  return check_launch("norm_partials");
}

int sbgm_groupnorm_apply(const void* x, size_t x_plane, const float* partials, int chunks, int pgroups, const float* gamma,
                         const float* beta, int groups, float eps, const void* skip, size_t skip_plane,
                         const float* tproj, int tproj_stride, int act, void* y, size_t y_plane, int fmt,
                         int n, int hw, int c, void* stream) {
  SBGM_REQUIRE(c % 8 == 0 && c <= 2048 && groups >= 1 && c % groups == 0 && chunks >= 1 && pgroups >= groups && pgroups % groups == 0,
               "groupnorm_apply: bad c=%d groups=%d pgroups=%d chunks=%d", c, groups, pgroups, chunks);
  const int vecs = c / 8;
  const size_t smem2 = (static_cast<size_t>(c) + groups) * 2 * sizeof(float);
  int slots = 148 * 8;
  SBGM_DISPATCH_FMT(fmt, (slots = resident_blocks(reinterpret_cast<const void*>(gn_apply_kernel<FMT>), 256, smem2)));
  const int per_n_blocks = max(1, min(ceil_div(static_cast<long long>(hw) * vecs, 256 * 4), slots / max(n, 1)));
  dim3 g2(per_n_blocks, n);
  SBGM_DISPATCH_FMT(fmt, (launch_k((gn_apply_kernel<FMT>), g2, 256, smem2, as_stream(stream), 
                             x, x_plane, partials, chunks, pgroups, gamma, beta, groups, eps, skip, skip_plane, tproj,
                             tproj_stride, act, y, y_plane, hw, c)));
  return check_launch("groupnorm_apply");
}

int sbgm_layernorm(const void* x, size_t x_plane, const float* gamma, const float* beta, float eps,
                   void* y, size_t y_plane, int fmt, int rows, int c, void* stream) {
  SBGM_REQUIRE(c % 8 == 0 && c <= 512, "layernorm: c=%d must be a multiple of 8 and <= 512", c);
  SBGM_DISPATCH_FMT(fmt, (launch_k((layernorm_kernel<FMT>), ceil_div(rows, 8), 256, 0, as_stream(stream), 
                             x, x_plane, gamma, beta, eps, y, y_plane, rows, c)));
  return check_launch("layernorm");
}

int sbgm_upsample2x(const void* x, size_t x_plane, void* y, size_t y_plane, int fmt, int n, int h, int w, int c,
                    void* stream) {
  SBGM_REQUIRE(c % 8 == 0, "upsample2x: c=%d must be a multiple of 8", c);
  const size_t total = static_cast<size_t>(n) * h * w * (c / 8);
  SBGM_REQUIRE(total < (1ull << 32), "upsample2x: tensor too large for 32-bit indexing");
  SBGM_DISPATCH_FMT(fmt, (launch_k((upsample2x_kernel<FMT>), grid_for(total, 256), 256, 0, as_stream(stream), 
                             x, x_plane, y, y_plane, n, h, w, c)));
  return check_launch("upsample2x");
}

int sbgm_stem_im2col(const float* x, const float* planes, int np, int cc, int c_begin, int c_end, void* out, size_t out_plane,
                     int fmt, int n, int h, int w, void* stream) {
  SBGM_REQUIRE(h % 2 == 0 && w % 2 == 0, "stem_im2col: h=%d and w=%d must be even", h, w);
  SBGM_REQUIRE(c_begin >= 0 && c_end > c_begin && c_end <= cc + 1, "stem_im2col: bad channel range [%d, %d) of %d", c_begin, c_end, cc + 1);
  SBGM_REQUIRE(c_end <= 1 || (planes != nullptr && (np == 1 || np == n)), "stem_im2col: conditioning planes missing or batch %d != 1, %d", np, n);
  const int nch = c_end - c_begin;
  SBGM_REQUIRE(static_cast<long long>(n) * nch <= 65535 && h / 2 <= 65535, "stem_im2col: grid too large");
  dim3 grid(ceil_div(w / 2, 32), h / 2, n * nch);
  SBGM_DISPATCH_FMT(fmt, (launch_k((stem_im2col_kernel<FMT>), grid, 256, 0, as_stream(stream), x, planes, np, cc, c_begin, nch, out,
                                   out_plane, n, h, w)));
  return check_launch("stem_im2col");
}

int sbgm_final_conv(const void* in, size_t in_plane, int fmt, const float* weight, const float* bias,
                    const float* inv_std, int inv_std_stride, int inv_std_step_stride, const int32_t* step_counter,
                    float* out, int n, int h, int w, int cin, int cout, void* stream) {
  SBGM_REQUIRE(cin % 8 == 0 && cout >= 1 && cout <= 4, "final_conv: cin=%d cout=%d unsupported", cin, cout);
  const size_t smem = static_cast<size_t>(cout) * 9 * cin * sizeof(float);
  SBGM_REQUIRE(smem <= 48 * 1024, "final_conv: weights exceed shared memory");
  const size_t npix = static_cast<size_t>(n) * h * w;
  const int grid = grid_for(npix * 32, 256, 148 * 8);
  cudaStream_t st = as_stream(stream);
#define SBGM_FC(CO) \
  SBGM_DISPATCH_FMT(fmt, (launch_k((final_conv_kernel<FMT, CO>), grid, 256, smem, st, in, in_plane, weight, bias, inv_std, inv_std_stride, inv_std_step_stride, step_counter, out, n, h, w, cin)))
  switch (cout) {
    case 1: SBGM_FC(1); break;
    case 2: SBGM_FC(2); break;
    case 3: SBGM_FC(3); break;
    default: SBGM_FC(4); break;
  }
#undef SBGM_FC
  return check_launch("final_conv");
}

int sbgm_final_gather(const float* proj, const float* bias, const float* inv_std, int inv_std_stride,
                      int inv_std_step_stride, const int32_t* step_counter, float* out, int n, int h, int w,
                      void* stream) {
  const size_t total = static_cast<size_t>(n) * h * w;
  launch_k((final_gather_kernel), grid_for(total, 256), 256, 0, as_stream(stream), proj, bias, inv_std, inv_std_stride,
                                                                           inv_std_step_stride, step_counter, out, n, h, w);
  return check_launch("final_gather");
}

}  // extern "C"
