// conv_grad_simt.cu -- CUDA-core gradient kernels of the convolutions (any format, any stride / kernel size):
//   * data gradient (gather form) and weight gradient (split over pixels, deterministic two-stage) of a generic
//     NHWC convolution -- the strict-fp32 path, the cross-check of the tensor-core gradients (conv_wgrad_tc.cu,
//     conv_tc.cu in dgrad mode) and the fall-back for shapes those do not take;
//   * weight gradient of the encoder stem (Encoder.conv1, 8x8 stride 2 over NCHW fp32 planes, score_unet.py:310);
//   * backward of the final 64 -> 1 convolution fused with the 1/std scaling (score_unet.py:713-730, :879).
// In the reference all of these are cuDNN calls made by torch autograd.
#include "common.cuh"

namespace sbgm {

// ---- dgrad: dx[n,iy,ix,ci] = sum_{r,s,co} dy[n,oy,ox,co] * w[tap][co][ci],  oy*stride + r - pad = iy ----------
template <int FMT>
__global__ void dgrad_simt_kernel(const void* __restrict__ dy, size_t dy_plane, const float* __restrict__ wgt, void* __restrict__ dx,
                                  size_t dx_plane, int accumulate, int n, int h, int w, int cin, int cout, int kh, int kw,
                                  int stride, int pad, int ho, int wo) {
  pdl_grid_sync();
  const int vecs = cin >> 3;
  const size_t total = static_cast<size_t>(n) * h * w * vecs;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int vec = static_cast<int>(i % vecs);
    size_t r0 = i / vecs;
    const int ix = static_cast<int>(r0 % w);
    r0 /= w;
    const int iy = static_cast<int>(r0 % h);
    const int b = static_cast<int>(r0 / h);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < kh; ++r) {
      const int ty = iy + pad - r;
      if (ty < 0 || ty % stride != 0) continue;
      const int oy = ty / stride;
      if (oy >= ho) continue;
      for (int s = 0; s < kw; ++s) {
        const int tx = ix + pad - s;
        if (tx < 0 || tx % stride != 0) continue;
        const int ox = tx / stride;
        if (ox >= wo) continue;
        const size_t opix = (static_cast<size_t>(b) * ho + oy) * wo + ox;
        const float* wt = wgt + (static_cast<size_t>(r) * kw + s) * cout * cin + vec * 8;
        for (int co = 0; co < cout; co += 8) {
          float g[8];
          Act<FMT>::load8(dy, dy_plane, opix * cout + co, g);
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(wt + static_cast<size_t>(co + k) * cin));
            const float4 w1 = __ldg(reinterpret_cast<const float4*>(wt + static_cast<size_t>(co + k) * cin) + 1);
            acc[0] = fmaf(g[k], w0.x, acc[0]); acc[1] = fmaf(g[k], w0.y, acc[1]); acc[2] = fmaf(g[k], w0.z, acc[2]); acc[3] = fmaf(g[k], w0.w, acc[3]);
            acc[4] = fmaf(g[k], w1.x, acc[4]); acc[5] = fmaf(g[k], w1.y, acc[5]); acc[6] = fmaf(g[k], w1.z, acc[6]); acc[7] = fmaf(g[k], w1.w, acc[7]);
          }
        }
      }
    }
    if (accumulate) {
      float old[8];
      Act<FMT>::load8(dx, dx_plane, i * 8, old);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += old[j];
    }
    Act<FMT>::store8(dx, dx_plane, i * 8, acc);
  }
}

// ---- wgrad: ws[split][co][tap*cin + ci] = sum over the split's output pixels of dy[p][co] * x[p*stride + tap - pad][ci] ----
template <int FMT>
__global__ void __launch_bounds__(256)
wgrad_simt_kernel(const void* __restrict__ x, size_t x_plane, const void* __restrict__ dy, size_t dy_plane, float* __restrict__ ws,
                  int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, int ho, int wo, int ci_blocks,
                  int pix_per_split) {
  pdl_grid_sync();
  __shared__ float xs[16][64];
  __shared__ float ds[16][64];
  const int cib = blockIdx.x % ci_blocks, cob = blockIdx.x / ci_blocks;
  const int tap = blockIdx.y, r = tap / kw, s = tap - r * kw;
  const int split = blockIdx.z;
  const size_t npix = static_cast<size_t>(n) * ho * wo;
  const size_t p_begin = static_cast<size_t>(split) * pix_per_split;
  const size_t p_end = min(npix, p_begin + pix_per_split);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lp = (threadIdx.x & 127) >> 3, lv = threadIdx.x & 7;     // loader: pixel 0..15, vector 0..7
  const bool load_x = threadIdx.x < 128;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (size_t p0 = p_begin; p0 < p_end; p0 += 16) {
    const size_t p = p0 + lp;
    float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (p < p_end) {
      if (load_x) {
        const int ox = static_cast<int>(p % wo), oy = static_cast<int>((p / wo) % ho), b = static_cast<int>(p / (static_cast<size_t>(wo) * ho));
        const int iy = oy * stride + r - pad, ix = ox * stride + s - pad, ch = cib * 64 + lv * 8;
        if (iy >= 0 && iy < h && ix >= 0 && ix < w && ch < cin)
          Act<FMT>::load8(x, x_plane, ((static_cast<size_t>(b) * h + iy) * w + ix) * cin + ch, v);
      } else {
        const int ch = cob * 64 + lv * 8;
        if (ch < cout) Act<FMT>::load8(dy, dy_plane, p * cout + ch, v);
      }
    }
    __syncthreads();
    float* dst = load_x ? &xs[lp][lv * 8] : &ds[lp][lv * 8];
#pragma unroll
    for (int j = 0; j < 8; ++j) dst[j] = v[j];
    __syncthreads();
#pragma unroll
    for (int pp = 0; pp < 16; ++pp) {
      const float4 a = *reinterpret_cast<const float4*>(&ds[pp][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&xs[pp][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
  const size_t K = static_cast<size_t>(kh) * kw * cin;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = cob * 64 + ty * 4 + i;
    if (co >= cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ci = cib * 64 + tx * 4 + j;
      if (ci < cin) ws[(static_cast<size_t>(split) * cout + co) * K + static_cast<size_t>(tap) * cin + ci] = acc[i][j];
    }
  }
}

// Sum the split partials in a fixed order and emit torch's OIHW layout: out[co][ci][tap].
__global__ void wgrad_reduce_kernel(const float* __restrict__ ws, int splits, int cout, int taps, int cin, float* __restrict__ out) {
  pdl_grid_sync();
  const size_t K = static_cast<size_t>(taps) * cin;
  const size_t total = static_cast<size_t>(cout) * K;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int ci = static_cast<int>(i % cin);
    const int tap = static_cast<int>((i / cin) % taps);
    const size_t co = i / K;
    float acc = 0.0f;
    for (int z = 0; z < splits; ++z) acc += __ldg(ws + static_cast<size_t>(z) * total + i);
    out[(co * cin + ci) * taps + tap] = acc;
  }
}

// ---- stem wgrad --------------------------------------------------------------------------------------
// ws[chunk][ci][tap][co] = sum over the chunk's output pixels of df1[p][co] * in[n][ci][2 oy + r - 3][2 ox + s - 3]
constexpr int kStemChunks = 64;
template <int FMT>
__global__ void __launch_bounds__(256)
stem_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ planes, int np, int cc, const void* __restrict__ df, size_t df_plane,
                  float* __restrict__ ws, int n, int h, int w) {
  pdl_grid_sync();
  __shared__ float patch[8][64];
  __shared__ float g[8][64];
  const int chunk = blockIdx.x, ci = blockIdx.y;
  const int ho = h / 2, wo = w / 2;
  const size_t npix = static_cast<size_t>(n) * ho * wo;
  const size_t per = ((npix + kStemChunks - 1) / kStemChunks + 7) / 8 * 8;
  const size_t p_begin = chunk * per, p_end = min(npix, p_begin + per);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (size_t p0 = p_begin; p0 < p_end; p0 += 8) {
    __syncthreads();
    for (int item = threadIdx.x; item < 512; item += 256) {
      const int pp = item >> 6, tap = item & 63;
      const size_t p = p0 + pp;
      float v = 0.0f;
      if (p < p_end) {
        const int ox = static_cast<int>(p % wo), oy = static_cast<int>((p / wo) % ho), b = static_cast<int>(p / (static_cast<size_t>(wo) * ho));
        const int iy = 2 * oy + (tap >> 3) - 3, ix = 2 * ox + (tap & 7) - 3;
        if (iy >= 0 && iy < h && ix >= 0 && ix < w) {
          v = (ci == 0) ? x[(static_cast<size_t>(b) * h + iy) * w + ix]
                        : planes[((static_cast<size_t>(np == 1 ? 0 : b) * cc + (ci - 1)) * h + iy) * w + ix];
        }
      }
      patch[pp][tap] = v;
    }
    if (threadIdx.x < 64) {
      const int pp = threadIdx.x >> 3, vec = threadIdx.x & 7;
      const size_t p = p0 + pp;
      float v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (p < p_end) Act<FMT>::load8(df, df_plane, p * 64 + vec * 8, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) g[pp][vec * 8 + j] = v[j];
    }
    __syncthreads();
#pragma unroll
    for (int pp = 0; pp < 8; ++pp) {
      const float4 a = *reinterpret_cast<const float4*>(&patch[pp][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&g[pp][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
  float* dst = ws + ((static_cast<size_t>(chunk) * gridDim.y + ci) * 64) * 64;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) dst[(ty * 4 + i) * 64 + tx * 4 + j] = acc[i][j];
}
__global__ void stem_wgrad_reduce_kernel(const float* __restrict__ ws, int cin, float* __restrict__ out) {
  pdl_grid_sync();
  const int total = cin * 64 * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int co = i & 63, tap = (i >> 6) & 63, ci = i >> 12;
    float acc = 0.0f;
    for (int k = 0; k < kStemChunks; ++k) acc += ws[static_cast<size_t>(k) * total + i];
    out[(static_cast<size_t>(co) * cin + ci) * 64 + tap] = acc;
  }
}

// ---- stem dgrad: d(x || planes)[b][ci][iy][ix] = sum_{r,s,co} df[b][oy][ox][co] * w[co][ci][r][s],  2 oy + r - 3 = iy ------------
// Thread = one input pixel of one parity class (blockIdx.y): its 16 taps are r = 7 - py - 2 ky at df row jy + py - 2 + ky (same
// for the columns), so a warp's weight loads are uniform.  The fp32 path, and the cross-check of stem_dgrad_tc.cu.
template <int FMT>
__global__ void __launch_bounds__(128)
stem_dgrad_simt_kernel(const void* __restrict__ df, size_t df_plane, const float* __restrict__ w_oihw, float* __restrict__ dx,
                       float* __restrict__ dpl, int n, int cc, int h, int w) {
  pdl_grid_sync();
  const int hh = h / 2, wh = w / 2, cin = cc + 1;
  const int py = blockIdx.y >> 1, px = blockIdx.y & 1;
  const size_t total = static_cast<size_t>(n) * hh * wh;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int jx = static_cast<int>(i % wh), jy = static_cast<int>((i / wh) % hh), b = static_cast<int>(i / (static_cast<size_t>(wh) * hh));
    float acc[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) acc[c] = 0.0f;
    for (int ky = 0; ky < 4; ++ky) {
      const int oy = jy + py - 2 + ky, r = 7 - py - 2 * ky;
      if (oy < 0 || oy >= hh) continue;
      for (int kx = 0; kx < 4; ++kx) {
        const int ox = jx + px - 2 + kx, s = 7 - px - 2 * kx;
        if (ox < 0 || ox >= wh) continue;
        const size_t base = ((static_cast<size_t>(b) * hh + oy) * wh + ox) * 64;
        const float* wt = w_oihw + r * 8 + s;
        for (int v8 = 0; v8 < 8; ++v8) {
          float g[8];
          Act<FMT>::load8(df, df_plane, base + v8 * 8, g);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float* wc = wt + static_cast<size_t>(v8 * 8 + e) * cin * 64;
#pragma unroll
            for (int c = 0; c < 16; ++c)
              if (c < cin) acc[c] = fmaf(g[e], __ldg(wc + c * 64), acc[c]);
          }
        }
      }
    }
    const size_t hw = static_cast<size_t>(h) * w, pix = static_cast<size_t>(2 * jy + py) * w + 2 * jx + px;
    if (dx) dx[b * hw + pix] = acc[0];
    if (dpl) {
#pragma unroll
      for (int c = 1; c < 16; ++c)
        if (c < cin) dpl[(static_cast<size_t>(b) * cc + c - 1) * hw + pix] = acc[c];
    }
  }
}
__global__ void batch_sum_kernel(const float* __restrict__ src, float* __restrict__ out, int n, size_t per) {
  pdl_grid_sync();
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < per; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float acc = 0.0f;
    for (int b = 0; b < n; ++b) acc += src[b * per + i];
    out[i] = acc;
  }
}

// ---- final convolution (cin -> 1, 3x3, pad 1) backward, fused with the 1/std scaling ---------------------
// g[n,y,x] = dscore[n,y,x] * inv_std[n]
template <int FMT>
__global__ void final_conv_bwd_input_kernel(const float* __restrict__ dscore, const float* __restrict__ inv_std, const float* __restrict__ wgt,
                                            void* __restrict__ da, size_t da_plane, int n, int h, int w, int cin) {
  pdl_grid_sync();
  extern __shared__ float wsm[];  // [9][cin]
  for (int i = threadIdx.x; i < 9 * cin; i += blockDim.x) wsm[i] = wgt[i];
  __syncthreads();
  const uint32_t vecs = cin >> 3;
  const uint32_t total = static_cast<uint32_t>(n) * h * w * vecs;      // < 2^32 (host-checked): 32-bit divisions only
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int vec = static_cast<int>(i % vecs);
    uint32_t r0 = i / vecs;
    const int x = static_cast<int>(r0 % w);
    r0 /= w;
    const int y = static_cast<int>(r0 % h);
    const int b = static_cast<int>(r0 / h);
    const float sc = inv_std ? inv_std[b] : 1.0f;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int oy = y - r + 1;
      if (oy < 0 || oy >= h) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int ox = x - s + 1;
        if (ox < 0 || ox >= w) continue;
        const float g = __ldg(dscore + (static_cast<size_t>(b) * h + oy) * w + ox) * sc;
        const float* wp = wsm + (r * 3 + s) * cin + vec * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = fmaf(g, wp[j], acc[j]);
      }
    }
    Act<FMT>::store8(da, da_plane, static_cast<size_t>(i) * 8, acc);
  }
}

// Both gradients in one pass over the activation (cin = 64, 128 or 256): a block owns tiles of kFinalTileRows x lanes pixels
// of one image, stages g (zero outside the image: no boundary branches) for the tile + halo in shared memory, and each thread
// (pixel column `lane`, channel vector `vec`) walks the tile's rows: the SAME nine g values feed da[p][ci] += g * w[tap][ci] and
// dW[tap][ci] += g * a[p][ci]; it also sums da per channel (the bias gradient of the convolution that produced `a`).  Loads of
// `a` are issued four rows ahead.  Per block: warp-shuffle reduction over the pixel lanes, then one partial row.
// Algorithmic traffic: read a + write da (2 x n*h*w*cin elements) -- the two separate kernels read / wrote the same bytes at
// ~1/6 of the HBM rate (72 accumulators per thread, one load in flight, boundary branches).
constexpr int kFinalTileRows = 8;
template <int FMT>
__global__ void __launch_bounds__(256, 1)
final_conv_bwd_fused_kernel(const float* __restrict__ dscore, const float* __restrict__ inv_std, const void* __restrict__ a, size_t a_plane,
                            const float* __restrict__ wgt, void* __restrict__ da, size_t da_plane, float* __restrict__ partials,
                            int n, int h, int w, int cin) {
  pdl_grid_sync();
  extern __shared__ float sm[];
  const int vecs = cin >> 3, lanes = 256 / vecs;
  const int vec = threadIdx.x % vecs, lane = threadIdx.x / vecs;
  const int gw = lanes + 2;
  float* wsm = sm;                                  // [9][cin]
  float* gs = wsm + 9 * cin;                        // [kFinalTileRows + 2][gw]
  float* red = gs + (kFinalTileRows + 2) * gw;      // [8 warps][10 * cin + 1]
  const int outs = 10 * cin + 1;
  for (int i = threadIdx.x; i < 9 * cin; i += 256) wsm[i] = wgt[i];
  float acc[9][8], bup[8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.0f;
#pragma unroll
  for (int j = 0; j < 8; ++j) bup[j] = 0.0f;
  float bsum = 0.0f;
  const int tiles_x = (w + lanes - 1) / lanes, tiles_y = (h + kFinalTileRows - 1) / kFinalTileRows;
  const int ntiles = n * tiles_y * tiles_x;
  // g of a tile + halo: at most two values per thread (lanes <= 32, host-checked), fetched one tile AHEAD into registers so that
  // the load is in flight while the current tile is computed
  auto fetch_g = [&](int tile, float (&r)[2]) {
    const int tx = tile % tiles_x, ty = (tile / tiles_x) % tiles_y, b = tile / (tiles_x * tiles_y);
    const float sc = inv_std ? inv_std[b] : 1.0f;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = threadIdx.x + k * 256;
      const int yy = ty * kFinalTileRows - 1 + i / gw, xx = tx * lanes - 1 + i % gw;
      r[k] = (i < (kFinalTileRows + 2) * gw && yy >= 0 && yy < h && xx >= 0 && xx < w)
                 ? __ldg(dscore + (static_cast<size_t>(b) * h + yy) * w + xx) * sc : 0.0f;
    }
  };
  float gnext[2] = {0.0f, 0.0f};
  if (static_cast<int>(blockIdx.x) < ntiles) fetch_g(blockIdx.x, gnext);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int tx = tile % tiles_x, ty = (tile / tiles_x) % tiles_y, b = tile / (tiles_x * tiles_y);
    const int y0 = ty * kFinalTileRows, x0 = tx * lanes;
    __syncthreads();
    if (threadIdx.x < (kFinalTileRows + 2) * gw) gs[threadIdx.x] = gnext[0];
    if (threadIdx.x + 256 < (kFinalTileRows + 2) * gw) gs[threadIdx.x + 256] = gnext[1];
    __syncthreads();
    if (tile + static_cast<int>(gridDim.x) < ntiles) fetch_g(tile + gridDim.x, gnext);
    const int x = x0 + lane;
    if (x >= w) continue;            // (no barrier below this point inside the iteration)
    const int rows = min(kFinalTileRows, h - y0);
    const size_t base = ((static_cast<size_t>(b) * h + y0) * w + x) * cin + vec * 8;
    const size_t row_pitch = static_cast<size_t>(w) * cin;
    for (int ly0 = 0; ly0 < rows; ly0 += 4) {
      float v[4][8];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (ly0 + k < rows) Act<FMT>::load8(a, a_plane, base + (ly0 + k) * row_pitch, v[k]);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int ly = ly0 + k;
        if (ly >= rows) break;
        float o[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            // tap (r, s) pairs input pixel (y, x) with output pixel (y - r + 1, x - s + 1); gs origin is (y0 - 1, x0 - 1)
            const float g = gs[(ly - r + 2) * gw + lane - s + 2];
            const float4 w0 = *reinterpret_cast<const float4*>(wsm + (r * 3 + s) * cin + vec * 8);
            const float4 w1 = *reinterpret_cast<const float4*>(wsm + (r * 3 + s) * cin + vec * 8 + 4);
            o[0] = fmaf(g, w0.x, o[0]); o[1] = fmaf(g, w0.y, o[1]); o[2] = fmaf(g, w0.z, o[2]); o[3] = fmaf(g, w0.w, o[3]);
            o[4] = fmaf(g, w1.x, o[4]); o[5] = fmaf(g, w1.y, o[5]); o[6] = fmaf(g, w1.z, o[6]); o[7] = fmaf(g, w1.w, o[7]);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[r * 3 + s][j] = fmaf(g, v[k][j], acc[r * 3 + s][j]);
          }
        Act<FMT>::store8(da, da_plane, base + ly * row_pitch, o);
#pragma unroll
        for (int j = 0; j < 8; ++j) bup[j] += o[j];
        if (vec == 0) bsum += gs[(ly + 1) * gw + lane + 1];
      }
    }
  }
  // reduce over the pixel lanes of the warp (threads `vecs` apart share a channel vector), then over the 8 warps
  for (int off = vecs; off < 32; off <<= 1) {
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[t][j] += __shfl_xor_sync(0xffffffffu, acc[t][j], off);
#pragma unroll
    for (int j = 0; j < 8; ++j) bup[j] += __shfl_xor_sync(0xffffffffu, bup[j], off);
    bsum += __shfl_xor_sync(0xffffffffu, bsum, off);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, wl = threadIdx.x & 31;
  float* mine = red + static_cast<size_t>(warp) * outs;
  if (vecs >= 32) {                      // one pixel lane per warp: every thread holds distinct channels
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) mine[t * cin + vec * 8 + j] = acc[t][j];
#pragma unroll
    for (int j = 0; j < 8; ++j) mine[9 * cin + 1 + vec * 8 + j] = bup[j];
    if (vec == 0) mine[9 * cin] = bsum;
  } else if (wl < vecs) {                // after the butterfly every lane holds the warp total of its vector
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) mine[t * cin + vec * 8 + j] = acc[t][j];
#pragma unroll
    for (int j = 0; j < 8; ++j) mine[9 * cin + 1 + vec * 8 + j] = bup[j];
    if (vec == 0) mine[9 * cin] = bsum;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < outs; i += 256) {
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sum += red[static_cast<size_t>(k) * outs + i];
    partials[static_cast<size_t>(blockIdx.x) * outs + i] = sum;
  }
}
// finish of the fused kernel: dW (OIHW, O = 1), db, and the producing convolution's bias gradient dbias_up[cin] (nullable)
__global__ void final_conv_bwd_fused_finish_kernel(const float* __restrict__ partials, int blocks, int cin, float* __restrict__ dW,
                                                   float* __restrict__ db, float* __restrict__ dbias_up) {
  pdl_grid_sync();
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;    // one warp per output
  const int outs = 10 * cin + 1;
  if (i >= outs) return;
  float s = 0.0f;
  for (int k = lane; k < blocks; k += 32) s += partials[static_cast<size_t>(k) * outs + i];
  s = warp_sum(s);
  if (lane != 0) return;
  if (i < 9 * cin) {
    const int tap = i / cin, ci = i - tap * cin;
    dW[ci * 9 + tap] = s;
  } else if (i == 9 * cin) {
    db[0] = s;
  } else if (dbias_up) {
    dbias_up[i - 9 * cin - 1] = s;
  }
}

constexpr int kFinalBwdBlocks = 1184;   // 148 SMs x 8: the kernel is latency-bound at low occupancy (72 accumulators / thread)
template <int FMT>
__global__ void __launch_bounds__(256)
final_conv_bwd_weight_kernel(const float* __restrict__ dscore, const float* __restrict__ inv_std, const void* __restrict__ a, size_t a_plane,
                             float* __restrict__ partials, int n, int h, int w, int cin) {
  pdl_grid_sync();
  extern __shared__ float red[];   // [lanes][9 * cin + 1]
  const int vecs = cin >> 3, lanes = blockDim.x / vecs;
  const int vec = threadIdx.x % vecs, lane = threadIdx.x / vecs;
  const size_t npix = static_cast<size_t>(n) * h * w;
  float acc[9][8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[t][j] = 0.0f;
  float bsum = 0.0f;
  if (lane < lanes) {
    for (uint32_t p = blockIdx.x * lanes + lane; p < static_cast<uint32_t>(npix); p += gridDim.x * lanes) {    // 32-bit divisions
      const int x = static_cast<int>(p % w), y = static_cast<int>((p / w) % h), b = static_cast<int>(p / (static_cast<uint32_t>(w) * h));
      const float sc = inv_std ? inv_std[b] : 1.0f;
      float v[8];
      Act<FMT>::load8(a, a_plane, static_cast<size_t>(p) * cin + vec * 8, v);
      // a[p] is the input of output pixel (y - r + 1, x - s + 1) under tap (r, s)
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int oy = y - r + 1;
        if (oy < 0 || oy >= h) continue;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int ox = x - s + 1;
          if (ox < 0 || ox >= w) continue;
          const float g = __ldg(dscore + (static_cast<size_t>(b) * h + oy) * w + ox) * sc;
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[r * 3 + s][j] = fmaf(g, v[j], acc[r * 3 + s][j]);
        }
      }
      if (vec == 0) bsum += __ldg(dscore + p) * sc;
    }
    float* o = red + static_cast<size_t>(lane) * (9 * cin + 1);
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
      for (int j = 0; j < 8; ++j) o[t * cin + vec * 8 + j] = acc[t][j];
    if (vec == 0) o[9 * cin] = bsum;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 9 * cin + 1; i += blockDim.x) {
    float s = 0.0f;
    for (int l = 0; l < lanes; ++l) s += red[static_cast<size_t>(l) * (9 * cin + 1) + i];
    partials[static_cast<size_t>(blockIdx.x) * (9 * cin + 1) + i] = s;
  }
}
__global__ void final_conv_bwd_finish_kernel(const float* __restrict__ partials, int blocks, int cin, float* __restrict__ dW, float* __restrict__ db) {
  pdl_grid_sync();
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;    // one warp per output
  if (i > 9 * cin) return;
  float s = 0.0f;
  for (int k = lane; k < blocks; k += 32) s += partials[static_cast<size_t>(k) * (9 * cin + 1) + i];
  s = warp_sum(s);
  if (lane != 0) return;
  if (i == 9 * cin) { db[0] = s; return; }
  const int tap = i / cin, ci = i - tap * cin;
  dW[ci * 9 + tap] = s;     // OIHW with O = 1
}

static int cgrid_for(size_t items, int block, int max_blocks = 148 * 16) {
  size_t g = (items + block - 1) / block;
  if (g < 1) g = 1;
  if (g > static_cast<size_t>(max_blocks)) g = max_blocks;
  return static_cast<int>(g);
}

static void wgrad_simt_plan(int n, int ho, int wo, int cin, int cout, int taps, int* ci_blocks, int* co_blocks, int* splits, int* per) {
  *ci_blocks = ceil_div(cin, 64);
  *co_blocks = ceil_div(cout, 64);
  const long long npix = static_cast<long long>(n) * ho * wo;
  const long long base = static_cast<long long>(*ci_blocks) * *co_blocks * taps;
  long long s = (148 * 6 + base - 1) / base;
  const long long max_s = (npix + 63) / 64;
  if (s > max_s) s = max_s;
  if (s < 1) s = 1;
  if (s > 256) s = 256;
  long long pp = ((npix + s - 1) / s + 15) / 16 * 16;
  *splits = static_cast<int>((npix + pp - 1) / pp);
  *per = static_cast<int>(pp);
}

int stem_dgrad_batch_sum(const float* per_sample, float* out, int n, size_t per, cudaStream_t st) {
  launch_k((batch_sum_kernel), cgrid_for(per, 256), 256, 0, st, per_sample, out, n, per);
  return check_launch("stem_dgrad_batch_sum");
}

}  // namespace sbgm

using namespace sbgm;

extern "C" {

int sbgm_conv2d_dgrad_simt(const void* dy, size_t dy_plane, const float* weight_tap_co_ci, void* dx, size_t dx_plane, int accumulate,
                           int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, void* stream) {
  SBGM_REQUIRE(cin % 8 == 0 && cout % 8 == 0, "conv2d_dgrad_simt: cin=%d and cout=%d must be multiples of 8", cin, cout);
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  SBGM_REQUIRE(ho > 0 && wo > 0, "conv2d_dgrad_simt: empty output");
  const size_t total = static_cast<size_t>(n) * h * w * (cin / 8);
  SBGM_DISPATCH_FMT(fmt, (launch_k((dgrad_simt_kernel<FMT>), cgrid_for(total, 128, 148 * 32), 128, 0, as_stream(stream), 
                             dy, dy_plane, weight_tap_co_ci, dx, dx_plane, accumulate, n, h, w, cin, cout, kh, kw, stride, pad, ho, wo)));
  return check_launch("conv2d_dgrad_simt");
}

size_t sbgm_conv2d_wgrad_simt_workspace_floats(int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad) {
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  int cib, cob, splits, per;
  wgrad_simt_plan(n, ho, wo, cin, cout, kh * kw, &cib, &cob, &splits, &per);
  return static_cast<size_t>(splits) * cout * kh * kw * cin;
}

int sbgm_conv2d_wgrad_simt(const void* x, size_t x_plane, const void* dy, size_t dy_plane, float* dweight_oihw, int fmt, int n, int h,
                           int w, int cin, int cout, int kh, int kw, int stride, int pad, float* workspace, void* stream) {
  SBGM_REQUIRE(cin % 8 == 0 && cout % 8 == 0, "conv2d_wgrad_simt: cin=%d and cout=%d must be multiples of 8", cin, cout);
  const int ho = (h + 2 * pad - kh) / stride + 1, wo = (w + 2 * pad - kw) / stride + 1;
  SBGM_REQUIRE(ho > 0 && wo > 0, "conv2d_wgrad_simt: empty output");
  int cib, cob, splits, per;
  wgrad_simt_plan(n, ho, wo, cin, cout, kh * kw, &cib, &cob, &splits, &per);
  cudaStream_t st = as_stream(stream);
  dim3 grid(cib * cob, kh * kw, splits);
  SBGM_DISPATCH_FMT(fmt, (launch_k((wgrad_simt_kernel<FMT>), grid, 256, 0, st, x, x_plane, dy, dy_plane, workspace, n, h, w, cin, cout, kh, kw,
                                                                        stride, pad, ho, wo, cib, per)));
  const size_t total = static_cast<size_t>(cout) * kh * kw * cin;
  launch_k((wgrad_reduce_kernel), cgrid_for(total, 256), 256, 0, st, workspace, splits, cout, kh * kw, cin, dweight_oihw);
  return check_launch("conv2d_wgrad_simt");
}

int sbgm_wgrad_reduce(const float* workspace, int splits, int cout, int taps, int cin, float* dweight_oihw, void* stream) {
  const size_t total = static_cast<size_t>(cout) * taps * cin;
  launch_k((wgrad_reduce_kernel), cgrid_for(total, 256), 256, 0, as_stream(stream), workspace, splits, cout, taps, cin, dweight_oihw);
  return check_launch("wgrad_reduce");
}

size_t sbgm_stem_wgrad_workspace_floats(int cin) { return static_cast<size_t>(kStemChunks) * cin * 64 * 64; }

int sbgm_stem_wgrad(const float* x, const float* planes, int np, int cc, const void* df, size_t df_plane, int fmt, float* dweight_oihw,
                    int n, int h, int w, float* workspace, void* stream) {
  SBGM_REQUIRE(h % 2 == 0 && w % 2 == 0, "stem_wgrad: h=%d and w=%d must be even", h, w);
  SBGM_REQUIRE(cc == 0 || planes != nullptr, "stem_wgrad: conditioning planes missing");
  SBGM_REQUIRE(np == 1 || np == n, "stem_wgrad: planes batch %d must be 1 or %d", np, n);
  cudaStream_t st = as_stream(stream);
  const int cin = cc + 1;
  dim3 grid(kStemChunks, cin);
  SBGM_DISPATCH_FMT(fmt, (launch_k((stem_wgrad_kernel<FMT>), grid, 256, 0, st, x, planes, np, cc, df, df_plane, workspace, n, h, w)));
  launch_k((stem_wgrad_reduce_kernel), cgrid_for(static_cast<size_t>(cin) * 4096, 256), 256, 0, st, workspace, cin, dweight_oihw);
  return check_launch("stem_wgrad");
}

size_t sbgm_stem_dgrad_workspace_floats(int np, int cc, int n, int h, int w) {
  return np == 1 && n > 1 ? static_cast<size_t>(n) * cc * h * w : 0;
}

int sbgm_stem_dgrad_simt(const void* df, size_t df_plane, int fmt, const float* w_oihw, float* dx, float* dplanes, int np, int cc, int n,
                         int h, int w, float* workspace, void* stream) {
  SBGM_REQUIRE(h % 2 == 0 && w % 2 == 0 && h > 0 && w > 0, "stem_dgrad_simt: h=%d and w=%d must be even", h, w);
  SBGM_REQUIRE(cc >= 0 && cc < 16, "stem_dgrad_simt: %d conditioning channels (at most 15)", cc);
  SBGM_REQUIRE(np == 1 || np == n, "stem_dgrad_simt: planes batch %d must be 1 or %d", np, n);
  SBGM_REQUIRE(dplanes == nullptr || (cc > 0 && (np == n || n == 1 || workspace != nullptr)),
               "stem_dgrad_simt: dplanes needs cc > 0 and, for planes shared by the batch, a workspace");
  cudaStream_t st = as_stream(stream);
  const bool sum_batch = dplanes != nullptr && np == 1 && n > 1;
  float* dpl = sum_batch ? workspace : dplanes;
  const size_t total = static_cast<size_t>(n) * (h / 2) * (w / 2);
  dim3 grid(cgrid_for(total, 128, 148 * 8), 4);
  SBGM_DISPATCH_FMT(fmt, (launch_k((stem_dgrad_simt_kernel<FMT>), grid, 128, 0, st, df, df_plane, w_oihw, dx, dpl, n, cc, h, w)));
  const int rc = check_launch("stem_dgrad_simt");
  if (rc != 0 || !sum_batch) return rc;
  return stem_dgrad_batch_sum(workspace, dplanes, n, static_cast<size_t>(cc) * h * w, st);
}

static bool final_fused_ok(int cin) {       // 8, 16 or 32 channel vectors: 32, 16 or 8 pixel lanes, a g tile of <= 512 values
  const int vecs = cin / 8;
  return cin % 8 == 0 && vecs >= 8 && vecs <= 32 && (vecs & (vecs - 1)) == 0;
}
static int final_fused_blocks() { return 148; }   // persistent: one block per SM (249 registers x 256 threads)

size_t sbgm_final_conv_backward_scratch_floats(int cin) {
  const size_t fused = static_cast<size_t>(final_fused_blocks()) * (10 * cin + 1), split = static_cast<size_t>(kFinalBwdBlocks) * (9 * cin + 1);
  return fused > split ? fused : split;
}

int sbgm_final_conv_backward(const float* dscore, const float* inv_std, const void* a, size_t a_plane, int fmt,
                             const float* weight_tap_ci, void* da, size_t da_plane, float* dweight_oihw, float* dbias, float* dbias_up,
                             int n, int h, int w, int cin, float* scratch, void* stream) {
  SBGM_REQUIRE(cin % 8 == 0 && cin <= 256, "final_conv_backward: cin=%d unsupported", cin);
  cudaStream_t st = as_stream(stream);
  const int vecs = cin / 8, lanes = 256 / vecs;
  const size_t total = static_cast<size_t>(n) * h * w * vecs;
  SBGM_REQUIRE(total < (1ull << 32), "final_conv_backward: tensor too large for 32-bit indexing");
  if (final_fused_ok(cin)) {
    const size_t smem = (9 * cin + static_cast<size_t>(kFinalTileRows + 2) * (lanes + 2) + 8 * (10 * cin + 1)) * sizeof(float);
    const int blocks = final_fused_blocks();
    SBGM_DISPATCH_FMT(fmt, {
      auto kf = final_conv_bwd_fused_kernel<FMT>;
      if (smem > 48 * 1024 && cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess) {
        set_error("final_conv_backward: cannot reserve %zu bytes of shared memory", smem);
        return 1;
      }
      launch_k((kf), blocks, 256, smem, st, dscore, inv_std, a, a_plane, weight_tap_ci, da, da_plane, scratch, n, h, w, cin);
    });
    launch_k((final_conv_bwd_fused_finish_kernel), ceil_div((10 * cin + 1) * 32, 256), 256, 0, st, scratch, blocks, cin, dweight_oihw, dbias,
             dbias_up);
    return check_launch("final_conv_backward");
  }
  SBGM_REQUIRE(dbias_up == nullptr, "final_conv_backward: dbias_up needs cin = 64, 128 or 256 (cin=%d)", cin);
  const size_t smem_w = static_cast<size_t>(lanes) * (9 * cin + 1) * sizeof(float);
  SBGM_DISPATCH_FMT(fmt, {
    auto kw_ = final_conv_bwd_weight_kernel<FMT>;
    if (smem_w > 48 * 1024 && cudaFuncSetAttribute(kw_, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem_w)) != cudaSuccess) {
      set_error("final_conv_backward: cannot reserve %zu bytes of shared memory", smem_w);
      return 1;
    }
    launch_k((final_conv_bwd_input_kernel<FMT>), cgrid_for(total, 256), 256, 9 * cin * sizeof(float), st, dscore, inv_std, weight_tap_ci, da, da_plane, n, h, w, cin);
    launch_k((kw_), kFinalBwdBlocks, 256, smem_w, st, dscore, inv_std, a, a_plane, scratch, n, h, w, cin);
  });
  launch_k((final_conv_bwd_finish_kernel), ceil_div((9 * cin + 1) * 32, 256), 256, 0, st, scratch, kFinalBwdBlocks, cin, dweight_oihw, dbias);
  return check_launch("final_conv_backward");
}

}  // extern "C"
