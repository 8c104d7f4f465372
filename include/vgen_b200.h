/*
 * vgen_b200 -- C ABI of libvgen_b200.so: hand-written sm_100a kernels for the VGen sampling hot path
 * (DDIM loop -> spatio-temporal UNet forward -> AutoencoderKL decode).
 *
 * The reference (ali-vilab/VGen) is pure PyTorch and has no FFI for this path: every op below replaces
 * a torch/cuDNN/cuBLAS/xformers library call made from a reference nn.Module.  Each entry cites the
 * reference call site it stands in for (paths relative to the reference root).  The Python classes in
 * vgen_b200/ (registered under the reference's MODEL / DIFFUSION / AUTO_ENCODER registry names) are the
 * only callers; they bind this header with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: raw device pointers, sizes and a cudaStream_t passed as void*; no torch types.
 *   - activations are fp16, channels-last ("tokens x channels", NHWC / [f][h][w][c]); weights fp16,
 *     K-major [out][taps*in]; biases / norm affine fp32; all accumulation fp32.
 *   - every function returns 0 on success; otherwise vgen_last_error() describes the failure.
 *   - no hidden synchronisation, no allocation: the caller owns every buffer (incl. workspaces).
 *   - not thread-safe per stream; one process per GPU.
 */
#ifndef VGEN_B200_H_
#define VGEN_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VGEN_B200_ABI_VERSION 2

/* ---- library ---------------------------------------------------------------------------------- */
int vgen_abi_version(void);
const char* vgen_last_error(void);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches). */
int64_t vgen_launch_count(void);
/* tap-GEMM implementation: 0 = auto (default: tcgen05 CTA pairs, single CTA for one-tile problems),
 * 1 = SIMT cross-check kernel (debug), 2 = force 1-CTA tcgen05, 3 = force 2-CTA (cta_group::2) tcgen05. */
int vgen_set_tapgemm_impl(int impl);

/* ---- tap-GEMM family (tcgen05.mma + TMA; tapgemm_sm100.cu) ------------------------------------ */
typedef struct vgen_epilogue {
  float alpha;              /* accumulator scale (1.0f = none)                                        */
  const float* bias;        /* [n] fp32 or NULL                                                       */
  const void* group_bias;   /* fp16 [groups][n] or NULL: per-frame bias, added after fp16 rounding     */
  int64_t group_bias_ld;    /*   (ResBlock "h + emb_out": tools/modules/unet/util.py:909-919)          */
  int64_t group_bias_div;   /*   row = image_index / group_bias_div (frames per video); 0 or 1 = per image */
  const void* residual;     /* fp16 [rows][n] or NULL: added after fp16 rounding (skip / x_in adds)    */
  int64_t residual_ld;
  int geglu;                /* 1: out[rows][n/2] = value * gelu(gate); W rows interleaved per bn block */
  int bn;                   /* N tile (32..256, multiple of 32; GEGLU: multiple of 64); 0 = auto       */
  /* LayerNorm folded into the GEMM (vgen_linear only): with w = W * diag(gamma) (rounded to fp16), col_sum[n] =
   * sum_k w[n][k], bias = b + W beta and row_stats[r] = {rstd_r, -mean_r * rstd_r} (vgen_row_stats),
   *   LN(x) W^T + b  =  rstd_r * (x w^T)[r][n] + (-mean_r rstd_r) * col_sum[n] + bias[n]
   * so the normalised activations are never written (nn.LayerNorm -> nn.Linear, util.py:694-704,731-741).
   * Both NULL = off; GEGLU: col_sum is indexed like bias (packed weight rows). */
  const float* row_stats;   /* fp32 [rows][2] or NULL                                                  */
  const float* col_sum;     /* fp32 [n] or NULL                                                        */
} vgen_epilogue;

/* out[m][n] = epi(a[m][:k] . w[n][:k])       -- nn.Linear / 1x1 conv / Conv1d(k=1)
 * replaces: util.py:224-229 (to_q/k/v/out), :711 (GEGLU.proj), :736 (FF out), :338,:353 (proj_in/out),
 *           :1213,:1229 (Conv1d proj), autoencoder.py:344-363 (q/k/v/proj_out 1x1), :305 (nin_shortcut) */
int vgen_linear(const void* a, int64_t m, int64_t k, int64_t lda, const void* w, int64_t n, void* out,
                int64_t ldo, const vgen_epilogue* epi, void* stream);

/* 3x3 / stride 1 / pad 1 conv on [nimg][h][w][c] fp16; w is [n][9*c] with k = (ky*3+kx)*c + ci.
 * replaces: nn.Conv2d in ResBlock util.py:845-876, Upsample.conv :761, head unet_t2v.py:204-207,
 *           VAE ResnetBlock / Upsample / conv_in / conv_out autoencoder.py:282-300,448-452,603,647 */
int vgen_conv2d_3x3(const void* x, int64_t nimg, int64_t h, int64_t w_, int64_t c, const void* w, int64_t n,
                    void* out, int64_t ldo, const vgen_epilogue* epi, void* stream);

/* temporal (3,1,1) conv, pad (1,0,0), on [f][hw][c] fp16 (one video); w is [n][3*c], k = kt*c + ci.
 * replaces: nn.Conv3d in TemporalConvBlock_v2 util.py:1662-1680 */
int vgen_tconv3(const void* x, int64_t f, int64_t hw, int64_t c, const void* w, int64_t n, void* out,
                int64_t ldo, const vgen_epilogue* epi, void* stream);
/* the same for `batch` videos stored back to back ([batch][f][hw][c]); frames of different videos never mix */
int vgen_tconv3_batch(const void* x, int64_t batch, int64_t f, int64_t hw, int64_t c, const void* w, int64_t n,
                      void* out, int64_t ldo, const vgen_epilogue* epi, void* stream);

/* ---- normalisation (norm.cu; HBM-bound, fp32 statistics) ---------------------------------------- */
/* GroupNorm(32 groups) over x[n][p][c] fp16 (statistics per sample n over p*c/32 values), optional
 * SiLU, y fp16.  For the 5-D (all-frames-jointly) norms pass n = batch, p = f*h*w.
 * replaces: nn.GroupNorm(+nn.SiLU) util.py:845-849,867-869,329,1211,1663-1680; autoencoder.py:15-16 */
int64_t vgen_group_norm_workspace_bytes(int64_t n);
int vgen_group_norm(const void* x, void* y, int64_t n, int64_t p, int64_t c, const float* gamma, const float* beta,
                    float eps, int silu, void* workspace, void* stream);
/* LayerNorm over the last dim of x[rows][c] (row strides ldx / ldy).  replaces: nn.LayerNorm util.py:694-696,1429 */
int vgen_layer_norm(const void* x, void* y, int64_t rows, int64_t c, int64_t ldx, int64_t ldy, const float* gamma,
                    const float* beta, float eps, void* stream);

/* Statistics of that LayerNorm only: stats[rows][2] = {rstd, -mean * rstd} fp32 (two-pass mean / variance like
 * vgen_layer_norm; one read of x, 8 bytes written per row) for a GEMM with vgen_epilogue.row_stats.
 * replaces: the statistics half of nn.LayerNorm util.py:694-696 */
int vgen_row_stats(const void* x, int64_t rows, int64_t c, int64_t ldx, float eps, float* stats, void* stream);

/* ---- attention ---------------------------------------------------------------------------------- */
/* softmax(q k^T * scale) v, head_dim 64, no mask (attn_sm100.cu, tcgen05 + TMEM).  q[batch][lq][heads*64]
 * with token stride ldq (so q/k/v may be column slices of one fused projection buffer); k/v have
 * batch / kv_batch_div batches (a context shared by the frames of a video is stored once).
 * replaces: xformers.ops.memory_efficient_attention, util.py:254-259 (spatial self / cross attention) */
int vgen_attention_d64(const void* q, const void* k, const void* v, void* out, int64_t batch, int64_t heads,
                       int64_t lq, int64_t lk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo,
                       int64_t kv_batch_div, float scale, void* stream);
/* Single-head attention with head_dim 512 (attn_d512_sm100.cu, tcgen05 flash attention: the [lq, lk] score matrix
 * never leaves the SM): out[b][i][:] = softmax_j(q[b][i].k[b][j] * scale) v[b][j][:]; q/k/v/out rows of 512 fp16 with
 * row strides ld* (multiples of 8), batches lq*ld / lk*ld apart.
 * replaces: AttnBlock.forward of the SD VAE, autoencoder.py:365-389 (w_ = bmm(q,k) * c**-0.5; softmax; bmm(v, w_)) */
int vgen_attention_d512(const void* q, const void* k, const void* v, void* out, int64_t batch, int64_t lq, int64_t lk,
                        int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo, float scale, void* stream);
/* Same op through the instrumented twin kernel: per-phase cycle counters of one mid-grid CTA's softmax warps
 * (timing16: 16 int64: per q-tile {wait S, load+max, wait P buffer, exponentials+store, total, blocks}) -- diagnosis only
 * (tools/bench_attn.py; the numbers behind DESIGN.md's account of where the attention kernel's time goes) */
int vgen_attention_d64_debug(const void* q, const void* k, const void* v, void* out, int64_t batch, int64_t heads,
                             int64_t lq, int64_t lk, int64_t ldq, int64_t ldk, int64_t ldv, int64_t ldo,
                             int64_t kv_batch_div, float scale, long long* timing16, void* stream);
/* Per-pixel attention over L <= 32 frames (attn_temporal.cu, register-resident mma.sync): token t of
 * sequence s lives at q + s*seq_stride + t*tok_stride (+ head*head_dim).  head_dim 64 is the fast path;
 * any head_dim <= 64, L <= 64 is served by a scalar kernel (I2VGen's 4-channel local encoder).
 * Videos back to back in one launch: sequence s is pixel (s % seqs_per_batch) of video (s / seqs_per_batch), whose
 * base is q + video*batch_stride (seqs_per_batch <= 0: one video, batch strides ignored).
 * replaces: memory_efficient_attention in TemporalTransformer util.py:1258-1261; Attention util.py:1396-1424 */
int vgen_attention_temporal(const void* q, const void* k, const void* v, void* out, int64_t nseq, int64_t heads,
                            int64_t L, int64_t head_dim, int64_t tok_stride, int64_t seq_stride,
                            int64_t tok_stride_o, int64_t seq_stride_o, int64_t seqs_per_batch, int64_t batch_stride,
                            int64_t batch_stride_o, float scale, void* stream);
/* in-place softmax(x * scale) over rows of x[rows][n] fp16 (VAE AttnBlock, autoencoder.py:377-379) */
int vgen_softmax_rows(void* x, int64_t rows, int64_t n, int64_t ld, float scale, void* stream);

/* ---- data movement / pointwise (elementwise.cu) ------------------------------------------------- */
/* x[n][c][p] (fp32 or fp16) -> y[n][p][c_pad] fp16 (extra channels zero): 'b c f h w -> (b f) h w c' */
int vgen_cp_to_pc(const void* x, int x_is_f32, void* y, int64_t n, int64_t c, int64_t p, int64_t c_pad, void* stream);
/* x[n][p][ldx] fp16 (first c channels) -> y[n][c][p] (fp16 or fp32) */
int vgen_pc_to_cp(const void* x, int64_t ldx, void* y, int y_is_f32, int64_t n, int64_t c, int64_t p, void* stream);
/* channels-last im2col with zero padding (optionally SiLU on the gathered input); columns beyond
 * kh*kw*c up to kpad are zero.  Serves stride-2 / tiny-channel convs (Downsample util.py:946, first
 * conv unet_t2v.py:112, I2VGen conditioning convs unet_i2vgen.py:116-132, VAE conv_in) via vgen_linear */
int vgen_im2col(const void* x, void* out, int64_t nimg, int64_t h, int64_t w, int64_t c, int64_t kh, int64_t kw,
                int64_t stride, int64_t pad_t, int64_t pad_l, int64_t ho, int64_t wo, int64_t kpad, int act_silu,
                void* stream);
/* F.interpolate(scale_factor=2, mode='nearest') on [nimg][h][w][c] (util.py:768, autoencoder.py:455) */
int vgen_upsample_nearest2x(const void* x, void* y, int64_t nimg, int64_t h, int64_t w, int64_t c, void* stream);
/* dst[r][0:cols] = src[r][0:cols] with row strides (torch.cat along channels, unet_t2v.py:269) */
int vgen_copy2d(const void* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int64_t cols, void* stream);
/* op: 0 silu(a), 1 a+b, 2 gelu(a), 3 a*s, 4 a+s*b  (fp16, fp32 math) */
int vgen_eltwise(int op, const void* a, const void* b, void* y, int64_t n, float s, void* stream);
/* out = [gelu](silu_in?(a) @ w^T + bias) [+ res] for small m or tiny k (time / fps / context MLPs
 * unet_t2v.py:93-104, ResBlock emb_layers util.py:857-863, TransformerV2 linears util.py:1396-1452) */
int vgen_linear_small(const void* a, int64_t m, int64_t k, int64_t lda, const void* w, const float* bias, int64_t n,
                      const void* res, int64_t ldr, void* out, int64_t ldo, int silu_in, int gelu_out, void* stream);
/* sinusoidal_embedding util.py:178-190: out[b][dim] fp16 = cat[cos, sin](t * 10000^(-i/half)) */
int vgen_sinusoidal_embedding(const float* t, void* out, int64_t b, int64_t dim, void* stream);
/* nn.AdaptiveAvgPool2d on channels-last input, optional SiLU on the input (unet_i2vgen.py:128-129) */
int vgen_adaptive_avgpool(const void* x, void* y, int64_t nimg, int64_t h, int64_t w, int64_t c, int64_t oh, int64_t ow,
                          int silu_in, void* stream);

/* ---- condition adapters (cond_adapter.cu) ------------------------------------------------------- */
/* Stem of every VideoComposer condition adapter, unet_videolcm.py:296-302 (and :306-371, unet_tf2tv.py likewise):
 * Conv2d(cin -> cout, 3x3, pad 1) -> SiLU -> AdaptiveAvgPool2d((oh, ow)) per frame, fused (mma.sync tensor cores; the
 * full-resolution activation never leaves shared memory).  x: the condition in the reference layout [b][cin][f][h][w],
 * contiguous, fp32 (x_is_f32 = 1) or fp16; cin 1..4.  wt: fp16 K-major [cout][round_up(9*cin, 16)] with
 * k = (ky*3 + kx)*cin + ci, padded columns zero; bias fp32 [cout]; cout 8..64 in steps of 8.  out: fp16 channels-last
 * [(b f)][oh][ow][cout].  Pool bins are PyTorch's adaptive ones; a bin may span at most 16 rows / 32 columns. */
int vgen_cond_stem(const void* x, int x_is_f32, int64_t b, int64_t cin, int64_t f, int64_t h, int64_t w, const void* wt,
                   const float* bias, int64_t cout, int64_t oh, int64_t ow, void* out, void* stream);
/* `concat = concat + adapter_i(...)` over the adapters of one forward (unet_videolcm.py:598-699): out[r][c] =
 * fp16(sum_i srcs[i][r][c]) with the sum in fp32, in the order given (1..8 fp16 sources, row stride ld_src). */
int vgen_cond_sum(const void* const* srcs, int nsrc, int64_t rows, int64_t cols, int64_t ld_src, void* out, int64_t ld_out,
                  void* stream);

/* DiagonalGaussianDistribution.sample * scale_factor (autoencoder.py:85-90,211-225): moments fp16 [n][p][2*zc]
 * (mean | logvar, channels-last) + fp32 noise [n][zc][p] -> fp32 z [n][zc][p] */
int vgen_vae_sample(const void* moments, const float* noise, float* z, int64_t n, int64_t zc, int64_t p, float scale,
                    void* stream);

/* ---- model-variant prologues (variants.cu; SURVEY.md section 8 row a21) -------------------------- */
/* softmax(q k^T * scale) v for any head_dim <= 256 and ragged (lq, lk); same addressing as
 * vgen_attention_d64.  Serves the 16-token context transformer of UNetSD_HiGen (head_dim 160) and the CLIP towers
 * (77 causal text tokens, head_dim 64; 257 image tokens, head_dim 80).
 * replaces: CrossAttention / memory_efficient_attention inside TextContextCrossTransformerMultiLayer,
 * unet_higen.py:154-172 (BasicTransformerBlock util.py:674-741) */
int vgen_attention_cross_small(const void* q, const void* k, const void* v, void* out, int64_t batch, int64_t heads,
                               int64_t lq, int64_t lk, int64_t head_dim, int64_t ldq, int64_t ldk, int64_t ldv,
                               int64_t ldo, int64_t kv_batch_div, int causal, float scale, void* stream);
/* CLIP conditioning (clip_embedder.py:183-212 on open_clip's CLIP): causal = 1 above is the text tower's attn_mask.
 * out[r][:] = fp16(table[ids[r]][:] + pos[r % L][:]) -- token_embedding(text) + positional_embedding (:190-191) */
int vgen_embed_tokens(const int64_t* ids, const float* table, const float* pos, void* out, int64_t nrows, int64_t L,
                      int64_t W, int64_t vocab, void* stream);
/* x[b][i] = fp16(x[b][i] + add[i]), i < n: "x = x + self.positional_embedding" of the vision tower
 * (utils/reward/open_clip/transformer.py VisionTransformer.forward) */
int vgen_add_rows_f32(void* x, const float* add, int64_t batch, int64_t n, void* stream);
/* F.interpolate(x.transpose(1,2), size=lout, mode='linear').transpose(1,2) on x[nseq][lin][c] fp16
 * (motion embedding, unet_higen.py:389-392) */
int vgen_interp_linear_rows(const void* x, void* y, int64_t nseq, int64_t lin, int64_t lout, int64_t c, void* stream);
/* Fourier_filter(x, threshold=1, scale) of unet_sr600.py:30-49 on channels-last x[nimg][h][w][ldx] (first c
 * channels), written to y[nimg][h][w][ldy]: the four centre bins of the shifted spectrum are scaled. */
int vgen_fourier_lowfreq_filter(const void* x, int64_t ldx, void* y, int64_t ldy, int64_t nimg, int64_t h, int64_t w,
                                int64_t c, float scale, void* stream);
/* UpsampleSR600 (util.py:792-804): nearest x2, keeping output rows [row0, row0+rows_out) of the 2h rows */
int vgen_upsample_nearest2x_rows(const void* x, void* y, int64_t nimg, int64_t h, int64_t w, int64_t c, int64_t row0,
                                 int64_t rows_out, void* stream);
/* dst[r][0:cols] = fp16(src[r][0:cols] * s) with row strides ("x[:, :C/2] *= 1.1", unet_sr600.py:272-273,279) */
int vgen_scale_copy2d(const void* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int64_t cols, float s,
                      void* stream);

/* ---- sampler ------------------------------------------------------------------------------------ */
/* One fused DDIM update (diffusion_ddim.py:157-162 CFG mix, :194-196 v->x0 | :190-192 eps->x0, :230-240):
 *   out = u + g*(y-u) in fp16 (u NULL: out = y); x0; eps; xt <- c4*x0 + c5*eps (+ c6*noise).
 * coef7 = {sqrt_ab[t], sqrt(1-ab[t]), sqrt(1/ab[t]), sqrt(1/ab[t]-1), sqrt(ab_prev), sqrt(1-ab_prev-sigma^2),
 *          sigma*mask} as fp32 (the host keeps the fp64 tables; timestep/index math is bit-exact there).
 * x0_out (may be NULL) receives the predicted x0, the second value ddim_sample returns (:241). */
int vgen_ddim_step(float* xt, const void* y, const void* u, const float* noise, int64_t n, float guide_scale,
                   const float* coef7, int mean_type_v, float* x0_out, void* stream);

/* GaussianDiffusion (diffusion_gauss.py), the SR600 sampler pair -- sampler_gauss.cu.
 * out[b][n_per] = u + guide_scale*(y-u) in fp16 (:206-210) and stats[b][4] = {sum y, sum y^2, sum out, sum out^2}
 * (fp64, zeroed by the call) for the std-ratio rescale of arXiv:2305.08891 (:212-218). */
int vgen_cfg_combine(const void* y, const void* u, void* out, int64_t batch, int64_t n_per, float guide_scale,
                     double* stats, void* stream);
/* x0 prediction (:220-230) from the fp32 latent xt and the fp16 model output `out`.  stats != NULL applies
 * out *= guide_rescale*std(y)/std(out) + (1-guide_rescale) first.  pred_type: 0 x0, 1 eps, 2 v;
 * alpha/sigma are the table entries of the (batch-uniform) timestep. */
int vgen_gauss_x0(const float* xt, const void* out, const double* stats, float guide_rescale, float alpha, float sigma,
                  int pred_type, float* x0, int64_t batch, int64_t n_per, void* stream);
/* out = a0*x0 + a1*x1 + a2*x2 + a3*x3 (fp32; x1..x3 may be NULL; out may alias an input): model-input
 * scaling (:113), DPM-Solver++(2M) SDE update (:124-139), DDIM inversion step (:408-410) */
int vgen_lincomb_f32(float* out, int64_t n, const float* x0, float a0, const float* x1, float a1, const float* x2,
                     float a2, const float* x3, float a3, void* stream);

/* ---- video write-out ----------------------------------------------------------------------------- */
/* utils/video_op.py:180-192 (save_i2vgen_video_safe; same arithmetic in save_t2vhigen_video_safe :276-288 and
 * save_video_local :226-240): out[f][h][w][3] = uint8(trunc(clamp(video[c][f][h][w]*std[c] + mean[c], 0, 1) * 255)),
 * i.e. mul_, add_, clamp_, *255, 'c f h w -> f h w c', numpy astype('uint8') -- bit-exact, on the device, so frames
 * cross PCIe as bytes.  band_count (may be NULL; f entries, zeroed by the call) receives per frame the number of
 * output bytes in [117, 137]: the last-frame anomaly test of :199-201 (ratio > 0.4 drops the frame). */
int vgen_video_to_rgb8(const float* video, int64_t c, int64_t f, int64_t h, int64_t w, const float* mean3,
                       const float* std3, uint8_t* out, unsigned long long* band_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VGEN_B200_H_ */
