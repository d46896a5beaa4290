/* sbgm_b200.h -- C ABI of the B200-native (sm_100a) kernels behind the SBGM_DANRA hot path.
 *
 * The reference (TheaQG/SBGM_DANRA) has no FFI of its own: its hot path is three Python files
 * whose arithmetic is library calls (cuDNN / cuBLAS / ATen).  Every entry point below replaces
 * one of those call sites; the reference location is cited per function as file:line relative
 * to the reference root.  The host side (sbgm_danra_b200/*.py) mirrors the reference's Python
 * API and reaches these symbols through ctypes -- see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _host; `stream` is a cudaStream_t
 *   - all functions are asynchronous on `stream` and return 0 on success, non-zero on failure
 *     (sbgm_last_error() gives the message); nothing here falls back to the CPU
 *   - activations are NHWC ("pixels x channels"), C % 8 == 0, in one of four storage formats:
 *       SBGM_FMT_F32     float32
 *       SBGM_FMT_BF16    bfloat16
 *       SBGM_FMT_BF16X2  two bfloat16 planes hi|lo with x ~= hi + lo (16 significant bits);
 *                        the lo plane starts `plane` elements after the hi plane.  Tensor-core
 *                        products use hi*hi + lo*hi + hi*lo, i.e. fp32-class accuracy at
 *                        bf16 tensor throughput / 3.
 *       SBGM_FMT_F16     ONE float16 plane (11 significant bits, saturating stores).  Tensor-core layers in
 *                        this format take their WEIGHTS as two float16 planes  w_hi | w_lo * 2^11  (22
 *                        significant bits; `w_plane` = distance between them): the product is
 *                        x * w_hi + 2^-11 (x * w_lo') -- two tensor-core products, one activation plane --
 *                        so the only rounding left is the activations' (score rel-L2 2-5e-4 against the
 *                        reference's fp32, inside the 1e-3 gate; "fp16x2" in the Python API).  Inference only.
 *   - `plane` arguments are the hi->lo plane distance in elements (ignored unless BF16X2)
 */
#ifndef SBGM_B200_H_
#define SBGM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { SBGM_FMT_F32 = 0, SBGM_FMT_BF16 = 1, SBGM_FMT_BF16X2 = 2, SBGM_FMT_F16 = 3 };
#define SBGM_F16_WLO_SCALE 2048.0f   /* w_lo plane of an F16-format weight is stored times 2^11 (kept normal in float16) */
enum { SBGM_ACT_NONE = 0, SBGM_ACT_RELU = 1, SBGM_ACT_SILU = 2, SBGM_ACT_GELU = 3 };

const char* sbgm_last_error(void);
int sbgm_version(void);
/* 1 if the current device is compute capability 10.x (tcgen05 / TMEM / TMA present). */
int sbgm_device_is_sm100(void);

/* ---- layout / format ------------------------------------------------------------------- */
/* NCHW fp32 (the reference's tensor layout, score_unet.py:247-364) -> NHWC `fmt`, and back.  */
int sbgm_nchw_to_nhwc(const float* src, void* dst, size_t dst_plane, int fmt, int n, int c, int h, int w, void* stream);
int sbgm_nhwc_to_nchw(const void* src, size_t src_plane, int fmt, float* dst, int n, int c, int h, int w, void* stream);
/* fp32 <-> fmt on a flat buffer of `count` elements (count % 8 == 0); used to pack weights.   */
int sbgm_convert(const void* src, size_t src_plane, int src_fmt, void* dst, size_t dst_plane, int dst_fmt,
                 size_t count, void* stream);

/* ---- time embedding + projections -------------------------------------------------------
 * SinusoidalEmbedding.forward (score_unet.py:41-45), label embedding add (:307-308) and the nine
 * SiLU->Linear time projections (Encoder :373-383 used at :314-357; DecoderBlock :501-504,:609).
 *   t                            time of row r = t[r * t_row_stride + step * t_step_stride], where
 *                                step = *step_counter (0 if step_counter is NULL).  A sampler passes its
 *                                step table with t_row_stride = 0, t_step_stride = SBGM_STEP_COLS.
 *   y[rows] or NULL              class label per row (int64), added to embedding set 0 only
 *   fourier_w[n_sets][te/2]      the Gaussian-Fourier W buffers (set 0 = encoder, 1.. = decoder blocks)
 *   label_emb[n_cls+1][te]       or NULL
 *   proj_w[c_total][te], proj_b[c_total], proj_set[c_total] (which W set feeds output channel c)
 *   out[rows][c_total]           fp32
 */
int sbgm_time_embed_project(const float* t, int t_row_stride, int t_step_stride, const int32_t* step_counter,
                            const int64_t* y, const float* fourier_w, int n_sets, int te,
                            const float* label_emb, const float* proj_w, const float* proj_b,
                            const int32_t* proj_set, int c_total, float* out, int rows, void* stream);

/* SinusoidalEmbedding.forward alone (score_unet.py:41-45): out[rows][2*half] = cat(sin, cos)(2 pi t W). */
int sbgm_fourier_embed(const float* t, const float* fourier_w, int half, float* out, int rows, void* stream);

/* im2col of the stem's 8x8 stride-2 pad-3 window: out[n][oy][ox][(c - c_begin) * 64 + r * 8 + s] = in[n][c][2oy+r-3][2ox+s-3]
 * (0 outside), in = x || planes (channel 0 = x), out NHWC `fmt` with (c_end - c_begin) * 64 channels.  The stem then is a
 * 1x1 tensor-core convolution over this tensor (sbgm_conv2d_tc / _ex) and its weight gradient sbgm_conv2d_wgrad_tc. */
int sbgm_stem_im2col(const float* x, const float* planes, int np, int cc, int c_begin, int c_end, void* out, size_t out_plane,
                     int fmt, int n, int h, int w, void* stream);
/* Encoder.conv1 restricted to the noisy-field channel, on the tensor cores with the 8x8 stride-2 windows built in shared memory
 * (no im2col tensor in HBM):  out[n][oy][ox][co] = sum_{r,s} x[n][2oy+r-3][2ox+s-3] w[co][r*8+s] + partial[..][oy][ox][co] + tproj[n][co].
 *   x[n][h][w] fp32; w_packed [planes][64][64] K-major in the weight storage of `fmt` (planes `w_plane` apart);
 *   partial[partial_n][h/2][w/2][64] in `fmt`: the conditioning channels' contribution (sbgm_stem_conv), partial_n == 1
 *   broadcasts it over the batch, NULL = none; tproj[n][tproj_stride] fp32 or NULL; out NHWC `fmt`.  h % 16 == 0, w % 32 == 0. */
int sbgm_stem_x_tc(const float* x, const void* w_packed, size_t w_plane, const void* partial, size_t partial_plane, int partial_n,
                   const float* tproj, int tproj_stride, void* out, size_t out_plane, int fmt, int n, int h, int w, void* stream);
/* ---- stem convolution (Encoder.conv1, score_unet.py:206-211,:312-315) ---------------------
 * 8x8 stride-2 pad-3 convolution over the virtual channel concat  x || planes  (:273-291) for
 * the input-channel range [c_begin, c_end), CUDA cores (K is tiny and the op is bandwidth bound).
 *   x[n][h][w]              channel 0 (the noisy HR field), may be NULL if c_begin > 0
 *   planes[np][cc][h][w]    NCHW conditioning channels 1..cc; np == 1 broadcasts over the batch
 *   w_packed[cin][64 taps][64]  fp32, tap-major (see pack_stem_weight in engine.py)
 *   addend[na][h/2][w/2][64] fp32 NHWC partial sums or NULL (na == 1 broadcasts)
 *   tproj[n][tproj_stride]  fp32 time projection added per (n, channel) or NULL
 *   out                     NHWC `fmt` [n][h/2][w/2][64]
 */
int sbgm_stem_conv(const float* x, const float* planes, int np, int cc, int c_begin, int c_end,
                   const float* w_packed, const float* addend, int na, const float* tproj, int tproj_stride,
                   void* out, size_t out_plane, int fmt, int n, int h, int w, void* stream);

/* ---- convolution as implicit GEMM -------------------------------------------------------
 * Replaces nn.Conv2d at every 3x3 / 1x1 / 8x8 site of the UNet (encoder BasicBlocks via
 * torchvision resnet.py:89-103, Encoder.conv2 score_unet.py:214-219, DecoderBlock.conv_up/conv
 * :472-489) and nn.Linear inside ImageSelfAttention (:112-148; a Linear is a 1x1 convolution
 * over tokens).  Epilogue order:  v = acc + bias[co];  v += residual[pix][co];  v = act(v);
 * v += tproj[n][co].
 *   in  [n][h][w][cin]   NHWC `fmt`;   out [n][ho][wo][cout] NHWC `fmt`
 *   weight: packed [planes][cout][kh*kw*cin] (K-major, k = (r*kw + s)*cin + ci), same fmt as `in`
 *           for the tensor-core path; fp32 [kh*kw*cin][cout] for the SIMT path.
 * sbgm_conv2d_tc   tcgen05.mma + TMEM accumulators + TMA (BF16 / BF16X2; cin % 64 == 0, cout % 64 == 0)
 * sbgm_conv2d_simt fp32 CUDA-core implicit GEMM (F32; exact-arithmetic mode and debugging aid)
 */
int sbgm_conv2d_tc(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                   const void* residual, size_t res_plane, const float* tproj, int tproj_stride,
                   void* out, size_t out_plane, int fmt, int n, int h, int w, int cin, int cout,
                   int kh, int kw, int stride, int pad, int act,
                   const float* proj_w, int n_proj, float* proj_out,
                   void* workspace, size_t workspace_bytes, float* gn_partials, void* stream);
/* Fused GroupNorm statistics: if gn_partials != NULL (bias-only epilogue) the kernel also writes partial sums of
 * its output at 8-channel granularity, layout [n][chunks][cout/8][2] (sum, sum of squares), chunks =
 * sbgm_conv2d_tc_gn_chunks(...) (0 = this shape cannot fuse them).  Consumed by sbgm_groupnorm_apply. */
int sbgm_conv2d_tc_gn_chunks(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad);
/* Scratch for deterministic split-K (layers on 4x4 / 8x8 maps, where the output grid would leave most SMs
 * idle): 0 if the shape does not split.  Passing NULL / too little simply disables split-K. */
size_t sbgm_conv2d_tc_workspace_bytes(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw,
                                      int stride, int pad);
/* The same operator specialised for the 64 -> 64 channel 3x3 stride-1 convolutions that carry 45% of
 * the network's FLOPs (encoder layer1, decoder blocks 3 and final conv_up): a persistent kernel (one
 * CTA per SM) keeps the whole 9 x 64 x 64 weight tensor resident in shared memory, fetches each
 * input tile as three (rows+2)-high halo slabs that serve all nine taps (2.4x less L2->SM traffic
 * than per-tap boxes) and double-buffers the TMEM accumulator so the epilogue of one tile overlaps
 * the MMAs of the next.  Requires h % 8 == 0 and w % 16 == 0.  Extra outputs:
 *   proj_w / proj_out : as above
 *   gn_partials       : if non-NULL, per-(image, 32-pixel strip) GroupNorm partial sums of the stored
 *                       values at 8-channel granularity, layout [n][chunks][8][2] with chunks =
 *                       (h/8)*(w/16)*4, consumed by sbgm_groupnorm_apply (saves the statistics pass).
 */
int sbgm_conv3x3_c64(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                     const void* residual, size_t res_plane, const float* tproj, int tproj_stride,
                     void* out, size_t out_plane, int fmt, int n, int h, int w, int act,
                     const float* proj_w, int n_proj, float* proj_out, float* gn_partials, int gn_cpg, void* stream);
/* The same convolution over upsample2x(x), x = [n][h/2][w/2][64]: the bilinear F.interpolate(scale_factor=2, align_corners=False)
 * that opens every decoder block and the final layer (score_unet.py:560-570, :652-659) is produced inside the kernel's operand
 * stage (TMA loads the tile's low-resolution patch, producer warps interpolate the halo slab into the swizzled operand layout):
 * the 4x larger upsampled tensor is never written.  h, w are the OUTPUT (high-resolution) size; bias-only epilogue (act = none),
 * optionally with the projection or the GroupNorm statistics.  Single-plane formats only (SBGM_FMT_BF16, SBGM_FMT_F16). */
int sbgm_conv3x3_c64_up(const void* x, size_t x_plane, const void* weight, size_t w_plane, const float* bias, void* out,
                        size_t out_plane, int fmt, int n, int h, int w, int act, const float* proj_w, int n_proj,
                        float* proj_out, float* gn_partials, int gn_cpg, void* stream);
/* Projection epilogue (proj_w != NULL, cout == 64 only): instead of storing the 64 output channels the
 * kernel stores proj_out[pix][SBGM_PROJ_STRIDE] = sum_c v[c] * proj_w[q][c] for q < n_proj (fp32) -- the
 * nine per-tap partial products of the final 64 -> 1 convolution, so its input never touches HBM.
 * bias, tproj rows and proj_w must be 16-byte aligned. */
#define SBGM_PROJ_STRIDE 12
int sbgm_conv2d_simt(const float* in, const float* weight, const float* bias, const float* residual,
                     const float* tproj, int tproj_stride, float* out, int n, int h, int w, int cin, int cout,
                     int kh, int kw, int stride, int pad, int act, void* stream);

/* ---- normalisation ------------------------------------------------------------------------
 * GroupNorm / InstanceNorm of the decoder (score_unet.py:483-487, :582-590) fused with the
 * skip add, time-projection add and activation that follow norm2 (:593-613):
 *   y = act( (x - mean_g) * rstd_g * gamma[c] + beta[c] + skip[pix][c] + tproj[n][c] )
 * gamma/beta NULL = no affine (InstanceNorm2d); groups == c gives instance norm.
 * `partials` is scratch of sbgm_groupnorm_scratch_floats(n, c, h*w) floats.
 */
size_t sbgm_groupnorm_scratch_floats(int n, int c, int hw);
int sbgm_groupnorm(const void* x, size_t x_plane, const float* gamma, const float* beta, int groups, float eps,
                   const void* skip, size_t skip_plane, const float* tproj, int tproj_stride, int act,
                   void* y, size_t y_plane, int fmt, int n, int hw, int c, float* partials, void* stream);
/* The apply half alone, from partial sums [n][chunks][pgroups][2] produced by a convolution epilogue;
 * pgroups (a multiple of groups, c/8 for the fused statistics) consecutive partial groups form one group. */
int sbgm_groupnorm_apply(const void* x, size_t x_plane, const float* partials, int chunks, int pgroups, const float* gamma,
                         const float* beta, int groups, float eps, const void* skip, size_t skip_plane,
                         const float* tproj, int tproj_stride, int act, void* y, size_t y_plane, int fmt,
                         int n, int hw, int c, void* stream);
/* LayerNorm over the channel axis of [rows][c] tokens (ImageSelfAttention.ln1/ln2, :127-128). */
int sbgm_layernorm(const void* x, size_t x_plane, const float* gamma, const float* beta, float eps,
                   void* y, size_t y_plane, int fmt, int rows, int c, void* stream);

/* act( LayerNorm(x; gamma, beta, eps) W^T + b ) over token rows x[rows][cin] -> y[rows][cout] with the LayerNorm folded into the
 * tensor-core GEMM (ImageSelfAttention: ln1 -> mha.in_proj, ln2 -> ff.0 + GELU; score_unet.py:139-146).  `weight` holds
 * W diag(gamma) packed for `fmt`, `bias` = b + W beta, `colsum[cout]` the row sums of the packed weight:
 *     y = rstd_t (x W'^T - mean_t colsum) + b'
 * The per-token mean / rstd are computed inside the kernel from the operand tiles as they pass through shared memory; the
 * normalised tensor is never written.  act: SBGM_ACT_NONE or SBGM_ACT_GELU.  Tensor-core formats only. */
int sbgm_linear_ln_tc(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                      const float* colsum, float eps, void* out, size_t out_plane, int fmt, int rows, int cin, int cout,
                      int act, void* stream);

/* The attention half of ImageSelfAttention.forward (score_unet.py:139-143) in one launch, single-plane tensor-core formats
 * (SBGM_FMT_F16, SBGM_FMT_BF16):   out = x + out_proj( concat_h softmax(Q_h K_h^T / sqrt(d)) V_h ) + bias
 *   qkv[b*s][3c]  packed in_proj output (q | k | v), x[b*s][c] the block input (residual), w_out the packed out_proj weight
 *   ([planes][c][c] K-major; two float16 planes hi | lo * 2^11 in SBGM_FMT_F16, `w_plane` apart), bias[c] fp32, out[b*s][c].
 * Scores, probabilities and the per-head outputs never leave the SM (tcgen05 products with TMEM accumulators).
 * sbgm_attention_out_proj_supported: 1 for d = c / heads in {32, 64}, c in {128, 256} and s = 256 or s | 128. */
int sbgm_attention_out_proj_supported(int fmt, int b, int s, int c, int heads);
int sbgm_attention_out_proj(const void* qkv, const void* x, const void* w_out, size_t w_plane, const float* bias, void* out,
                            int fmt, int b, int s, int c, int heads, void* stream);

/* ---- bilinear x2 upsample (nn.Upsample(scale_factor=2, bilinear, align_corners=False),
 *      score_unet.py:467, :583) --------------------------------------------------------------- */
int sbgm_upsample2x(const void* x, size_t x_plane, void* y, size_t y_plane, int fmt, int n, int h, int w, int c,
                    void* stream);

/* ---- multi-head self-attention core (nn.MultiheadAttention inside ImageSelfAttention,
 *      score_unet.py:124,:141): out = softmax(Q K^T / sqrt(d)) V per head, from the packed
 *      in_proj output qkv[b][s][3c] (q | k | v), d = c / heads.  out[b][s][c]. ---------------- */
int sbgm_attention(const void* qkv, size_t qkv_plane, void* out, size_t out_plane, int fmt,
                   int b, int s, int c, int heads, void* stream);

/* ---- final convolution (Decoder.final_layer.conv, score_unet.py:713-730) fused with the
 *      division by the marginal std (ScoreNet.forward :876-877):
 *      out[n][co][h][w] = (conv3x3(in)[co] + bias[co]) * s_n             (NCHW fp32, cout <= 4)
 *      s_n = inv_std[n * inv_std_stride + step * inv_std_step_stride], step = *step_counter (0 if NULL);
 *      inv_std NULL = no scaling.  weight fp32 [cout][9][cin]. --------------------------------- */
int sbgm_final_conv(const void* in, size_t in_plane, int fmt, const float* weight, const float* bias,
                    const float* inv_std, int inv_std_stride, int inv_std_step_stride, const int32_t* step_counter,
                    float* out, int n, int h, int w, int cin, int cout, void* stream);
/* Second half of the fused final convolution: gathers the per-tap partial products written by the
 * projection epilogue, out[n][0][y][x] = (sum_{r,s} proj[n][y+r-1][x+s-1][3r+s] + bias) * s_n
 * (zero outside the image = the convolution's zero padding). */
int sbgm_final_gather(const float* proj, const float* bias, const float* inv_std, int inv_std_stride,
                      int inv_std_step_stride, const int32_t* step_counter, float* out, int n, int h, int w,
                      void* stream);

/* ---- counter-based noise + fused sampler updates -------------------------------------------
 * Noise stream: Philox4x32-10, key = seed, counter = (elem/4, draw); see oracle/philox_ref.py
 * for the exact definition (the oracle restates it in numpy).  `first_elem` is the index of
 * out[0] in the *global* [members][1][h][w] ensemble, so sharded ensembles are reproducible.
 */
int sbgm_philox_normal(float* out, size_t count, uint64_t seed, uint32_t draw, uint64_t first_elem, void* stream);
int sbgm_philox_uniform(float* out, size_t count, uint64_t seed, uint32_t draw, uint64_t first_elem, void* stream);

/* Per-step scalar table, one row of SBGM_STEP_COLS floats per sampler step (built on the host
 * with the reference's own arithmetic, score_sampling.py:96-103,169-176):
 *   [0] t   [1] g = sigma^t   [2] dt   [3] 1/std(t)   [4] g*g*dt   [5] noise scale
 *   (EM: sqrt(dt)*g, :125; PC predictor: sqrt(g*g*dt), :227)   [6..7] reserved
 * `step_counter` points at FOUR device int32 (the sampler state): [0] the current step, [1] scratch
 * (block-arrival count, zero), [2..3] the 64-bit Philox seed (lo, hi).  Kernels read row
 * step_counter[0]; the predictor / EM update increments it when its last block retires.  Keeping step
 * and seed on the device is what lets one captured CUDA graph (frozen kernel arguments) replay every
 * step of every sampler call.
 */
#define SBGM_STEP_COLS 8
/* x0 = z * std(1)  (score_sampling.py:93-95 / :167-168) */
int sbgm_sampler_init(float* x, size_t count, float std1, uint64_t seed, uint64_t first_elem, void* stream);
/* Euler-Maruyama / PC predictor update (score_sampling.py:124-125, :224-227):
 *   mean = x + (g*g*dt) * score ;  x = mean + noise_scale * z ;  ++*step_counter
 * draw id = draw_base + draw_stride * step.  `mean_out` receives `mean` (always written). */
int sbgm_sampler_predictor(float* x, const float* score, float* mean_out, size_t count, const float* step_table,
                           int32_t* step_counter, uint32_t draw_base, uint32_t draw_stride,
                           uint64_t first_elem, void* stream);
/* per-member sum of squares of `score` -> sumsq[members] (PC corrector, score_sampling.py:201) */
int sbgm_sampler_sumsq(const float* score, float* sumsq, int members, int per_member, void* stream);
/* Langevin corrector (score_sampling.py:198-204):  grad_norm = mean_b sqrt(sumsq[b]) over
 * `members_total` members (sumsq already holds every member of the global ensemble);
 *   eps = 2 (snr sqrt(per_member) / grad_norm)^2 ;  x += eps * score + sqrt(2 eps) * z          */
int sbgm_sampler_corrector(float* x, const float* score, const float* sumsq, int members_total, int per_member,
                           float snr, size_t count, const int32_t* step_counter,
                           uint32_t draw_base, uint32_t draw_stride, uint64_t first_elem, void* stream);
/* classifier-free guidance combine (guided_score_fn, score_sampling.py:54): out = (1+scale) s_c - scale s_u */
int sbgm_cfg_combine(const float* s_cond, const float* s_uncond, float scale, float* out, size_t count, void* stream);
/* copy row *step_counter of table[steps][cols] to out[cols] (time projections of the step) */
int sbgm_select_step_row(const float* table, int cols, const int32_t* step_counter, float* out, void* stream);

/* ---- back-transforms of sampled fields to physical units (SURVEY section 8(f), the step after the sampler) ------------
 * y = exp?(clamp?(scale * (x + pre_shift) + shift, lo, hi)): ZScoreBackTransform (sbgm/special_transforms.py:187-237),
 * ScaleBackTransform (:103-138) and every mode of PrcpLogBackTransform (:360-462) are instances. x and y may alias. */
int sbgm_back_transform(const float* x, float* y, size_t count, float pre_shift, float scale, float shift, float lo, float hi,
                        int do_clamp, int do_exp, void* stream);

/* y = back_transform(x) as above AND, per sample (n samples of `per` values), the numbers the reference's extreme-value
 * sentinel needs (sbgm/utils.py:1642-1671 report_precip_extremes: `torch.quantile(flat, 0.999, dim=1)`, `max`; driven by
 * sbgm/training.py:359-398 on the ground truth and :700-755 on generated fields):
 *   out[n][4] = { quantile `quantile` with linear interpolation (ATen's rank / lerp arithmetic), max, min, 0 }.
 * One block per sample, exact radix select in shared memory; x and y may alias. */
int sbgm_back_transform_extremes(const float* x, float* y, int n, int per, float pre_shift, float scale, float shift, float lo,
                                 float hi, int do_clamp, int do_exp, float quantile, float* out, void* stream);

/* ---- device-resident Dormand-Prince stages of ode_sampler (sbgm/score_sampling.py:239-300: scipy RK45 on the host) ----
 * State y[n], stages K[7][n] and results are float64 on the device; coefficient rows are HOST arrays (a row of the Butcher
 * tableau, at most 7 entries).
 *   combine   : out = y + h * sum_{s < n_stages} coef[s] K[s]   (out and/or its float32 copy out_f32, the network's input)
 *   rhs       : k_out = scale * score                           (dx/dt = -1/2 g(t)^2 score, :287-291)
 *   error_norm: *out_sumsq = sum_i ( h * sum_s coef[s] K[s][i] / (atol + max(|y_i|, |y_new_i|) * rtol) )^2, deterministic
 *               (y_new NULL: |y_i| alone -- the norms of scipy's select_initial_step with h = 1, coef = unit vector);
 *               scratch holds sbgm_rk45_scratch_doubles(n) doubles. */
int sbgm_rk45_combine(const double* y, const double* k_stages, size_t n, int n_stages, const double* coef_host, double h,
                      double* out, float* out_f32, void* stream);
int sbgm_rk45_rhs(const float* score, double scale, double* k_out, size_t n, void* stream);
size_t sbgm_rk45_scratch_doubles(size_t n);
int sbgm_rk45_error_norm(const double* k_stages, size_t n, int n_stages, const double* coef_host, double h, const double* y,
                         const double* y_new, double atol, double rtol, double* scratch, double* out_sumsq, void* stream);

/* ---- ensemble statistics (BASELINE.json parity criterion; evaluation itself is sbgm/evaluate_sbgm/, out of scope) ----
 * members[m][pixels] fp32 -> per-pixel mean, std (Bessel-corrected), and, given truth[pixels], the ensemble CRPS
 * E|X - y| - 1/2 E|X - X'| (crps may be NULL).  Lets a sampled ensemble be scored on the device before any D2H copy. */
int sbgm_ensemble_stats(const float* members, const float* truth, int m, size_t pixels, float* mean, float* stdev, float* crps,
                        void* stream);

/* ---- DSM loss (loss_fn, score_unet.py:936-985) -------------------------------------------
 * perturb: x_t = x + std[n] * z, z from the Philox stream (draw id `draw`), also stores z.
 * loss:    loss = 1/n * sum_{n,pix} w * (score * std[n] + z)^2, w = 0.5 sigmoid(sdf) + 0.5 or 1;
 *          two-stage deterministic reduction; `partials` has sbgm_dsm_scratch_floats(count) floats. */
int sbgm_dsm_perturb(const float* x, const float* std, float* xt, float* z, int n, int per_member, uint64_t seed,
                     uint32_t draw, uint64_t first_elem, void* stream);
size_t sbgm_dsm_scratch_floats(size_t count);
int sbgm_dsm_loss(const float* score, const float* std, const float* z, const float* sdf, int n, int per_member,
                  float* partials, float* loss_out, void* stream);

/* ==== training (DSM step): forward pieces with batch statistics + every backward =================
 * The reference obtains all of these from torch autograd (loss.backward(), sbgm/training.py:323-410)
 * over the modules of sbgm/score_unet.py; cuDNN/ATen supply the arithmetic.  Gradients of activations
 * use the same NHWC storage formats as the activations; parameter gradients are fp32 in torch's
 * parameter layouts (conv: OIHW).  All reductions are two-stage with a fixed order (deterministic). */

/* per (n, chunk) partial (sum, sumsq) over `groups` channel groups: partials[n][chunks][groups][2] with
 * chunks = sbgm_norm_partials_chunks(hw, c) (1..32).  groups == c gives the per-channel partials of train-mode
 * BatchNorm (torchvision resnet.py:89-103). */
int sbgm_norm_partials_chunks(int hw, int c);
int sbgm_norm_partials(const void* x, size_t x_plane, int fmt, int n, int hw, int c, int groups, float* partials, void* stream);
/* GroupNorm / InstanceNorm: stats[n][groups][2] = (mean, rstd) from partials[n][chunks][pgroups][2]
 * (the stand-alone partials above or the fused statistics of the convolution kernels). */
int sbgm_gn_stats_finalize(const float* partials, int chunks, int pgroups, int groups, int n, int hw, int c, float eps,
                           float* stats, void* stream);
/* BatchNorm2d.forward in training mode: stats[c][2] = (batch mean, rstd of the biased variance) and the
 * running_mean / running_var update (momentum, unbiased variance); either running pointer may be NULL. */
int sbgm_bn_stats_finalize(const float* partials, int chunks, int n, int hw, int c, float eps, float momentum, float* stats,
                           float* running_mean, float* running_var, void* stream);
/* y = act((x - mean) * rstd * gamma + beta + add + [tproj if tproj_pre_act]) + [tproj if !tproj_pre_act]
 * stats index: per_sample_stats == 1 ? [n][groups] : [groups] (BatchNorm: groups = c, per_sample_stats = 0;
 * per_sample_stats = 2: per-channel CONSTANT statistics, i.e. eval-mode BatchNorm -- its backward has no
 * mean / variance terms).
 * DecoderBlock.forward score_unet.py:559-627 (tproj before the activation); BasicBlock + Encoder.forward
 * :314-357 (ReLU, then the time projection). */
int sbgm_norm_apply(const void* x, size_t x_plane, const float* stats, int per_sample_stats, int groups, const float* gamma,
                    const float* beta, const void* add, size_t add_plane, const float* tproj, int tproj_stride,
                    int tproj_pre_act, int act, void* y, size_t y_plane, int fmt, int n, int hw, int c, void* stream);
/* backward of sbgm_norm_apply: dx, dadd (= gradient w.r.t. the pre-activation; NULL to skip), dgamma/dbeta[c]
 * (NULL for non-affine norms), dtproj[n][dtproj_stride] (NULL to skip), dbias_prev[c] (NULL to skip) = dx summed over
 * n and the pixels, i.e. the bias gradient of the convolution whose output x is (closed form from the reduction sums, no
 * extra pass).  Two launches: the reduction tree (last-block tickets, deterministic) and the apply pass.
 * `scratch`: sbgm_norm_backward_scratch_floats(n, c) floats, ZERO before its first use (its leading words are the
 * tickets; every launch leaves them zero again, so one zero-initialised buffer serves all layers of a stream).
 * Synchronised BatchNorm (data-parallel training with whole-batch statistics): call with stage = 1 (per-sample sums
 * [n][c][4] = sbgm_norm_backward_sums_floats(n, c) floats land at scratch + sbgm_norm_backward_sums_offset(n, c)),
 * all-gather those over the ranks, then stage = 2 with sums_all[n_all][c][4].  stage = 0 does everything locally
 * (sums_all = NULL). */
size_t sbgm_norm_backward_scratch_floats(int n, int c);
size_t sbgm_norm_backward_sums_offset(int n, int c);
size_t sbgm_norm_backward_sums_floats(int n, int c);
int sbgm_norm_backward(const void* dy, size_t dy_plane, const void* x, size_t x_plane, const float* stats, int per_sample_stats,
                       int groups, const float* gamma, const float* beta, const void* add, size_t add_plane,
                       const float* tproj, int tproj_stride, int tproj_pre_act, int act, void* dx, size_t dx_plane,
                       void* dadd, size_t dadd_plane, float* dgamma, float* dbeta, float* dbias_prev, float* dtproj, int dtproj_stride,
                       int fmt, int n, int hw, int c, float* scratch, int stage, const float* sums_all, int n_all, void* stream);
/* nn.LayerNorm backward (ImageSelfAttention.ln1 / ln2, score_unet.py:136-148) */
size_t sbgm_layernorm_backward_scratch_floats(int c);
int sbgm_layernorm_backward(const void* dy, size_t dy_plane, const void* x, size_t x_plane, const float* gamma, float eps,
                            void* dx, size_t dx_plane, float* dgamma, float* dbeta, int fmt, int rows, int c, float* scratch,
                            void* stream);
/* stand-alone activation (the feed-forward GELU keeps its pre-activation for the backward) */
int sbgm_act_forward(const void* x, size_t x_plane, void* y, size_t y_plane, int fmt, size_t count, int act, void* stream);
int sbgm_act_backward(const void* dy, size_t dy_plane, const void* x, size_t x_plane, void* dx, size_t dx_plane, int fmt,
                      size_t count, int act, void* stream);
/* dst += src (gradient accumulation where a tensor has several consumers) */
int sbgm_add_inplace(void* dst, size_t dst_plane, const void* src, size_t src_plane, int fmt, size_t count, void* stream);
/* out_per_sample[n][out_stride] (nullable) = sum over the hw pixels; out_total[c] (nullable) = sum over everything
 * (bias gradients; time-projection gradients of the encoder stages).  Total only: one launch (last-block ticket).
 * `scratch`: sbgm_channel_sums_scratch_floats(n, c) floats, ZERO before its first use (leading ticket words; every launch
 * leaves them zero again). */
size_t sbgm_channel_sums_scratch_floats(int n, int c);
int sbgm_channel_sums(const void* x, size_t x_plane, int fmt, int n, int hw, int c, float* out_per_sample, int out_stride,
                      float* out_total, float* scratch, void* stream);
/* adjoint of sbgm_upsample2x: dy [n, 2h, 2w, c] -> dx [n, h, w, c] */
int sbgm_upsample2x_backward(const void* dy, size_t dy_plane, void* dx, size_t dx_plane, int fmt, int n, int h, int w, int c,
                             void* stream);
/* attention core backward: dqkv [b*s][3c] from qkv, the forward's output `out` [b*s][c] (NULL: not available) and dout
 * [b*s][c].  bf16 with S % 16 == 0 and head dim 32 / 64 / 128 (and `out` given): ONE warp-level tensor-core launch, a CTA
 * per (image, head), nothing but dqkv written (attention_bwd_mma.cu).  Otherwise: fp32
 * batched CUDA-core GEMMs from `scratch` (..._scratch_floats floats; unused by the tensor-core path). */
size_t sbgm_attention_backward_scratch_floats(int b, int s, int c, int heads);
int sbgm_attention_backward(const void* qkv, size_t qkv_plane, const void* out, size_t out_plane, const void* dout, size_t dout_plane,
                            void* dqkv, size_t dqkv_plane, int fmt, int b, int s, int c, int heads, float* scratch, void* stream);
/* backward of sbgm_time_embed_project (one row per batch member): d_proj_w[c_total][te], d_proj_b[c_total],
 * d_label_emb[n_classes][te] (NULL when the model has no labels) */
size_t sbgm_time_embed_backward_scratch_floats(int n_sets, int te, int rows);
int sbgm_time_embed_backward(const float* dout, const float* t, const int64_t* y, const float* fourier_w, int n_sets, int te,
                             const float* label_emb, int n_classes, const float* proj_w, const int32_t* proj_set, int c_total,
                             int rows, float* d_proj_w, float* d_proj_b, float* d_label_emb, float* scratch, void* stream);

/* ---- convolution gradients --------------------------------------------------------------------
 * data gradient, CUDA cores: weight as fp32 [tap][cout][cin]; `accumulate` adds into dx */
int sbgm_conv2d_dgrad_simt(const void* dy, size_t dy_plane, const float* weight_tap_co_ci, void* dx, size_t dx_plane, int accumulate,
                           int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, void* stream);
/* generalised tensor-core convolution (data gradients = the forward implicit-GEMM kernel run over dy with flipped /
 * parity-sliced weights; ConvTranspose2d decoder; im2col stem): separate paddings, explicit logical output size and
 * scattered store out[n][oy*out_step+out_oy][ox*out_step+out_ox]; `residual` is read at the same positions
 * (accumulates an existing gradient) or, with res_pix_mod > 0, broadcast over the batch by pix % res_pix_mod. */
int sbgm_conv2d_tc_ex(const void* in, size_t in_plane, const void* weight, size_t w_plane, const float* bias,
                      const void* residual, size_t res_plane, int res_pix_mod, const float* tproj, int tproj_stride,
                      void* out, size_t out_plane, int fmt, int n, int h,
                      int w, int cin, int cout, int kh, int kw, int stride, int pad_h, int pad_w, int ho, int wo,
                      int out_h, int out_w, int out_step, int out_oy, int out_ox, int act, void* workspace,
                      size_t workspace_bytes, void* stream);
/* weight gradient -> dweight_oihw[cout][cin][kh][kw] fp32; x is the layer input [n,h,w,cin], dy [n,ho,wo,cout] */
size_t sbgm_conv2d_wgrad_simt_workspace_floats(int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad);
int sbgm_conv2d_wgrad_simt(const void* x, size_t x_plane, const void* dy, size_t dy_plane, float* dweight_oihw, int fmt, int n, int h,
                           int w, int cin, int cout, int kh, int kw, int stride, int pad, float* workspace, void* stream);
/* tensor cores (tcgen05, MN-major operands straight from the NHWC tensors; cin, cout multiples of 64) */
size_t sbgm_conv2d_wgrad_tc_workspace_floats(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad);
/* How sbgm_conv2d_wgrad_tc runs this shape (host only, launches nothing): plan[8] = {kernel (0 = per-unit, 1 = 3x3 halo slab),
 * output channels per CTA, pixel splits, tiles per split, total tiles, tile width, tile height, images per tile}.  Tiles are
 * numbered along the output width first, then its height, then the images; split s owns tiles [s * tiles per split, ...) and the
 * last split may be short.  Nonzero (sbgm_last_error) for a shape sbgm_conv2d_wgrad_tc rejects. */
int sbgm_conv2d_wgrad_tc_plan(int fmt, int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, int* plan);
int sbgm_conv2d_wgrad_tc(const void* x, size_t x_plane, const void* dy, size_t dy_plane, float* dweight_oihw, int fmt,
                         int n, int h, int w, int cin, int cout, int kh, int kw, int stride, int pad, float* workspace, void* stream);
/* sum workspace[splits][cout][taps*cin] over the splits in a fixed order into OIHW */
int sbgm_wgrad_reduce(const float* workspace, int splits, int cout, int taps, int cin, float* dweight_oihw, void* stream);
/* Encoder.conv1 (8x8 s2 p3 over NCHW fp32 x || planes, score_unet.py:310): weight gradient from df [n,h/2,w/2,64] */
size_t sbgm_stem_wgrad_workspace_floats(int cin);
int sbgm_stem_wgrad(const float* x, const float* planes, int np, int cc, const void* df, size_t df_plane, int fmt, float* dweight_oihw,
                    int n, int h, int w, float* workspace, void* stream);
/* Encoder.conv1 data gradient from df [n,h/2,w/2,64] (fmt): dx [n,1,h,w] and dplanes [np,cc,h,w], fp32 NCHW, each nullable;
 * np == 1 (planes shared by the batch): dplanes is the sum over the batch, built in `workspace` (the size below, 0 otherwise).
 * cc <= 15.  CUDA cores, any format, weight = conv1.weight as fp32 OIHW [64][cc+1][8][8]: */
size_t sbgm_stem_dgrad_workspace_floats(int np, int cc, int n, int h, int w);
int sbgm_stem_dgrad_simt(const void* df, size_t df_plane, int fmt, const float* w_oihw, float* dx, float* dplanes, int np, int cc, int n,
                         int h, int w, float* workspace, void* stream);
/* tensor cores (tcgen05), bf16 and split bf16: w_packed [4 parity classes (py * 2 + px)][planes][16][16 taps * 64] bf16, planes
 * w_plane elements apart, class c = sbgm_pack_weight(conv1.weight zero-padded to 16 input channels, transpose = 1, taps r * 8 + s
 * for r = 7 - py - 2 ky, s = 7 - px - 2 kx, ky and kx = 0..3 in that order) */
int sbgm_stem_dgrad_tc(const void* df, size_t df_plane, int fmt, const void* w_packed, size_t w_plane, float* dx, float* dplanes,
                       int np, int cc, int n, int h, int w, float* workspace, void* stream);
/* Decoder.final_layer.conv (cin -> 1, 3x3) + the 1/std scaling, backward: g = dscore * inv_std[n];
 * da [n,h,w,cin] (fmt), dweight_oihw[1][cin][3][3], dbias[1]; weight_tap_ci = fp32 [9][cin].  dbias_up[cin] (nullable) = da
 * summed over n,h,w: the bias gradient of the convolution that produced `a` (final_layer.conv_up), free in the same pass
 * (needs cin = 64, 128 or 256). */
size_t sbgm_final_conv_backward_scratch_floats(int cin);
int sbgm_final_conv_backward(const float* dscore, const float* inv_std, const void* a, size_t a_plane, int fmt,
                             const float* weight_tap_ci, void* da, size_t da_plane, float* dweight_oihw, float* dbias, float* dbias_up,
                             int n, int h, int w, int cin, float* scratch, void* stream);
/* Pack a torch OIHW fp32 weight for the tensor-core kernels in one launch: out[o][t][i] = w[co][ci][taps_host[t]]
 * with (o, i) = (co, ci), or (ci, co) when `transpose` (the flipped / parity-sliced data-gradient weights);
 * K-major bf16 or split-bf16 (planes `out_plane` elements apart).  taps_host is a HOST array of ntaps <= 64
 * flat tap indices r * kw + s.  A training step re-packs every parameter after each optimizer update. */
int sbgm_pack_weight(const float* w_oihw, int cout, int cin, int khw, const int* taps_host, int ntaps, int transpose,
                     void* out, size_t out_plane, int fmt, void* stream);
/* batched form of sbgm_pack_weight (ntaps <= 16 per job): all jobs in ceil(njobs / 80) launches; the job table is a
 * kernel parameter, so the call is capturable in a CUDA graph.  `jobs_host` is a HOST array. */
typedef struct {
  const float* w_oihw;
  void* out;
  size_t out_plane;
  int cout, cin, khw, ntaps, transpose;
  int taps[16];
} sbgm_pack_job;
int sbgm_pack_weights(const sbgm_pack_job* jobs_host, int njobs, int fmt, void* stream);
/* On-device batch assembly (sbgm/utils.py:405-480 `extract_samples`; the dataset transforms of sbgm/special_transforms.py:62-343
 * that sbgm/data_modules.py:727-997 applies on the CPU): ONE launch writes every float32 tensor of a batch from source tensors
 * of any dtype -- conversion, channel concatenation (a source lands at `dst_offset` inside each destination sample of
 * `dst_stride` elements; `inner` = elements per sample in the source) and the optional forward transform
 *     v = log ? log(x + eps) : x;   y = transform ? (((v - sub) * mul) / div) * post_mul + post_add : v.
 * jobs_dev: DEVICE table ordered by first_block; a block covers sbgm_batch_chunk_elems() elements of one job. */
enum { SBGM_DT_F32 = 0, SBGM_DT_F64 = 1, SBGM_DT_F16 = 2, SBGM_DT_BF16 = 3, SBGM_DT_I64 = 4, SBGM_DT_I32 = 5, SBGM_DT_I16 = 6,
       SBGM_DT_U8 = 7, SBGM_DT_I8 = 8 };
typedef struct {
  const void* src;
  float* dst;
  long long count, inner, dst_stride, dst_offset, first_block;
  int dtype, log, transform, pad_;
  float eps, sub, mul, div, post_mul, post_add;
} sbgm_batch_job;
int sbgm_batch_chunk_elems(void);
int sbgm_assemble_batch(const sbgm_batch_job* jobs_dev, int njobs, long long total_blocks, void* stream);
/* torch.optim.Adam / AdamW update (sbgm/training.py:407 `self.optimizer.step()`, optimizer built by sbgm/training_utils.py:672-698)
 * of EVERY parameter tensor in one launch.  chunks_dev: DEVICE table, one entry per block, each covering at most
 * sbgm_adam_chunk_elems() consecutive elements of one tensor.  Arithmetic follows torch/optim/adam.py (_single_tensor_adam,
 * amsgrad / maximize off): decoupled = 0 adds weight_decay * p to the gradient, 1 multiplies p by 1 - lr * weight_decay. */
typedef struct {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  int count;
  int pad_;
} sbgm_adam_chunk;
int sbgm_adam_chunk_elems(void);
int sbgm_adam_step(const sbgm_adam_chunk* chunks_dev, int n_chunks, double lr, double beta1, double beta2, float eps, float weight_decay,
                   int decoupled, double bias_correction1, double bias_correction2, void* stream);
/* d loss / d score of sbgm_dsm_loss, times *grad_loss (device scalar; NULL = 1) */
int sbgm_dsm_loss_backward(const float* score, const float* std, const float* z, const float* sdf, const float* grad_loss, int n,
                           int per_member, float* dscore, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SBGM_B200_H_ */
