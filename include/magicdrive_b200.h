/*
 * magicdrive_b200 — C ABI of the B200-native multi-view denoising hot path.
 *
 * Every entry point takes raw device pointers, sizes, strides and a cudaStream_t (as void*), returns 0 on
 * success or a negative status, and never allocates, synchronises or takes ownership.  mdb_last_error()
 * returns a thread-local message for the last failure.  Activations are bf16, channel-innermost (NHWC for
 * feature maps == [tokens, channels] for transformer blocks); accumulation is fp32.
 *
 * The reference has no native boundary of its own for this path except one op: xformers'
 * efficient_attention_forward_cutlass (third_party/xformers/xformers/csrc/attention/attention.cpp:27,
 * attention_forward_generic.cu:330-334).  Everything else it runs is a torch.nn call; each function below
 * names the reference call site (file:line under /root/reference) it replaces.
 */
#ifndef MAGICDRIVE_B200_H
#define MAGICDRIVE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDB_OK 0
#define MDB_ERR_INVALID (-1)
#define MDB_ERR_CUDA (-2)
#define MDB_ERR_UNSUPPORTED (-3)

const char* mdb_last_error(void);

/* Programmatic dependent launch for the launches that follow (process-wide flag, returns the previous value): the next
 * kernel's launch latency and prologue overlap the tail of its stream predecessor.  Switch it on only around
 * single-stream regions (the UNet up path); the environment variable MDB_PDL=0|1 overrides the flag. */
int mdb_set_pdl(int on);
int mdb_version(void);
/* 1 if a CUDA device of compute capability 10.x is usable, else 0 (never raises). */
int mdb_device_ok(void);

/* ------------------------------------------------------------------------------------------------
 * mdb_gemm_conv: tensor-core (tcgen05) GEMM / implicit-GEMM convolution with fused epilogue.
 *   out[pix, n] = scale * ( sum_{r,s,c} A[pix*stride + (r,s) - pad, c] * W[n, (r*taps_w+s)*C + c]
 *                           + bias[n] + rowbias[img(pix), n] ) + residual[pix, n]
 *   epi_mode 1 (GEGLU): W/bias are packed per 256-column tile as [128 value | 128 gate] and
 *   out[pix, j] = value_j * gelu(gate_j) with n_out/2 output columns.
 * Replaces: nn.Conv2d 3x3/1x1 in ResnetBlock2D (diffusers/models/resnet.py:537,560,586), Downsample2D
 * (resnet.py:199), Upsample2D.conv (resnet.py:129), Transformer2DModel.proj_in/proj_out
 * (transformer_2d.py:149,205), Attention.to_q/to_k/to_v/to_out (attention_processor.py:141-156),
 * GEGLU.proj + FeedForward out (attention.py:270,226), connector (magicdrive/networks/blocks.py:83),
 * ControlNet zero convs (magicdrive/networks/unet_addon_rawbox.py:221-272).
 * A may be split over two sources along channels (torch.cat skip connections, unet_2d_blocks.py:1984,2086).
 * Taps that fall outside the input read zeros on every side, so h_out / w_out may exceed the symmetric-pad size: the VAE
 * encoder's Downsample2D(padding=0) (resnet.py:215-220, F.pad(x, (0, 1, 0, 1)) then a stride-2 3x3 conv) is pad 0 with
 * h_out = (h_in - 2) / 2 + 1 (w_out likewise).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  const void* a0;      /* bf16 [n_img, h_in, w_in, lda0] using the first c0 channels */
  const void* a1;      /* optional second source (NULL if c1 == 0) */
  int c0, lda0, c1, lda1;
  int n_img, h_in, w_in;
  const void* w;       /* bf16 [n_out, taps_h*taps_w*(c0+c1)] */
  int n_out;
  int taps_h, taps_w, stride, pad_h, pad_w;
  int h_out, w_out;
  const float* bias;    /* [n_out] or NULL */
  const float* rowbias; /* [n_img, rowbias_ld] or NULL */
  int rowbias_ld;
  const void* residual; /* bf16 [pixels, ldr] or NULL */
  int ldr;
  void* out;            /* bf16 (or fp32 if out_is_f32) [pixels, ldo] */
  int ldo;
  int out_is_f32;
  float out_scale;
  int epi_mode;         /* 0 linear, 1 GEGLU */
  void* workspace;      /* split-K scratch (may be NULL => no split-K) */
  size_t workspace_bytes;
  int force_block_n;    /* 0 = auto; test hook */
  int force_splits;     /* 0 = auto; test hook */
  int kernel_variant;   /* 0 = auto (CTA-pair kernel where it applies, else the single-CTA split-K kernel); 2 = single-CTA
                         * persistent kernel; 3 = CTA-pair kernel; 4 = the pair kernel's code on single CTAs; test / A-B hook */
  int debug_flags;      /* ablation hook (0 in production): 1 skip stores, 2 skip epilogue loads, 4 skip TMEM loads */
  void* trace;          /* debug: device int64[8*16] receiving per-CTA clock64 stamps of the persistent kernel, or NULL */
  /* LayerNorm folded into the GEMM (attention.py:85,104,120; blocks.py:67-71): A is the RAW tensor x, W was
   * pre-multiplied by gamma (W' = W * gamma), bias holds c_n = sum_k beta_k W[n,k] + b_n, and the epilogue applies
   *   out = rstd_row * (acc - mean_row * ln_colsum[n]) + c_n
   * with mean/rstd from the per-row partial sums the PRODUCER of x wrote (stats_out of that call). */
  const float* ln_stats;   /* fp32 [pixels, ln_parts, 2] partial (sum, sum of squares) of the rows of A, or NULL */
  int ln_parts;
  float ln_eps;
  const float* ln_colsum;  /* fp32 [n_out]: sum_k W'[n, k] */
  /* Producer side: fp32 [pixels, mdb_gemm_conv_stats_parts(d), 2] receiving partial (sum, sum of squares) of every bf16
   * output row (after bias / residual), or NULL. */
  float* stats_out;
} mdb_gemm_desc;

int mdb_gemm_conv(const mdb_gemm_desc* d, void* stream);
/* Number of kernels mdb_gemm_conv would launch for this descriptor (1, or 2 with split-K). */
int mdb_gemm_conv_launches(const mdb_gemm_desc* d);
/* Partial-sum slots per output row that mdb_gemm_conv writes to stats_out for this descriptor (depends on the tiling the
 * planner picks); negative status if the descriptor cannot emit row statistics. */
int mdb_gemm_conv_stats_parts(const mdb_gemm_desc* d);

/* Direct (CUDA-core) convolution for tiny channel counts: conv_in 4->320 (unet_2d_condition.py:231),
 * conv_out 320->4 (:503), BEV map encoder (magicdrive/networks/map_embedder.py:66-76).
 * x: [n, h, w, cin] bf16 or fp32; w: fp32 [kh, kw, cin, cout] (output channel innermost: coalesced across a warp);
 * out bf16/fp32 [n, ho, wo, cout] (+= residual). */
int mdb_conv_direct(const void* x, int x_is_f32, int n, int h, int w, int cin, const float* wgt, const float* bias,
                    int cout, int kh, int kw, int stride_h, int stride_w, int pad_h, int pad_w, int ho, int wo,
                    int silu, const void* residual, void* out, int out_is_f32, void* stream);

/* GroupNorm (+SiLU) over NHWC, optionally over the channel-concat of two sources; writes one normalised tensor.
 * Replaces nn.GroupNorm + SiLU (resnet.py:535,556,598,630; transformer_2d.py:145; unet_2d_condition.py:492).
 * stats_ws: fp32 [max(n_img, 160) * groups * 2] scratch (per-image or per-CTA-run group partials). */
int mdb_groupnorm(const void* x0, int c0, int ld0, const void* x1, int c1, int ld1, int n_img, int hw, int groups,
                  float eps, const float* gamma, const float* beta, int silu, void* out, int ldo, float* stats_ws,
                  void* stream);

/* LayerNorm over the last dim of [rows, C] bf16 (attention.py:85,104,120; blocks.py:67-71). */
int mdb_layernorm(const void* x, long long rows, int c, int ldx, const float* gamma, const float* beta, float eps,
                  void* out, int ldo, void* stream);

/* Row softmax of fp32 scores into bf16 probabilities: out[r, j] = softmax_j(s[r, :cols]) for j < cols and 0 for
 * cols <= j < cols_out (K padding of the following P.V GEMM).  Used by the VAE decoder's single-head 512-wide attention
 * (unet_2d_blocks.py:433-446; attention_processor.py:1252), whose QK^T and PV products run on mdb_gemm_conv. */
int mdb_softmax_rows(const float* s, int lds, long long rows, int cols, void* out, int ldo, int cols_out, void* stream);

/* Fused multi-head attention forward, softmax(Q K^T * scale) V, bf16 in/out, fp32 softmax.
 * q: [b, Lq, heads*d] with row stride ldq; k, v: [b_kv, Lk, heads*d] with row strides ldk, ldv; out like q (ldo).
 * kv_index: device int32 [b * n_sets] of K/V batch indices (< b_kv) or NULL (then b_kv == b and batch i attends to
 * K/V batch i).  b_kv > b is the view-sharded case: K/V of all views were all-gathered, queries are local.
 * With n_sets == 2 the kernel computes
 *   out[b] = attn(q[b], kv[kv_index[2b]]) + attn(q[b], kv[kv_index[2b+1]])
 * which is the cross-view "add" mode (magicdrive/networks/blocks.py:112-121, 213-217) without the 2x token
 * duplication.  Replaces xformers efficient_attention_forward_cutlass / F.scaled_dot_product_attention
 * (attention_processor.py:1165-1171, 1252). */
int mdb_attention(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* out, int ldo, int b,
                  int b_kv, int heads, int lq, int lk, int d, const int* kv_index, int n_sets, float scale, void* stream);

/* The same with the K/V batches spread over n_src (1..3) buffers: k[i] / v[i] are [b_kv[i], Lk, heads*d] with row strides
 * ldk[i] / ldv[i]; kv_index entries are (source << 24) | batch index inside that source.  This is how the view-sharded mode
 * consumes its ring neighbours' K/V without gathering them: source 1 / 2 are the neighbour GPUs' K/V buffers, mapped through
 * NVLink peer memory (the TMA loads go over NVLink tile by tile, overlapping the local QK^T / PV work). */
int mdb_attention_multi(const void* q, int ldq, int n_src, const void* const* k, const int* ldk, const void* const* v,
                        const int* ldv, const int* b_kv, void* out, int ldo, int b, int heads, int lq, int lk, int d,
                        const int* kv_index, int n_sets, float scale, void* stream);

/* Debug hook (NULL in production): a device int64[3 * 16 * 8] buffer that receives clock64 stamps of the first CTA of
 * every following fused-attention launch (MMA warp and two softmax warps, 16 KV iterations, 8 points each);
 * tools/bench_attn.py --trace prints them.  Pass NULL to switch it off. */
int mdb_attention_debug_trace(void* device_i64_384);

/* out = a + b (bf16), n elements (unet_2d_condition_multiview.py:464-473, 487-488). */
int mdb_add(const void* a, const void* b, void* out, long long n, void* stream);

/* Nearest-neighbour resize NHWC, src index = floor(dst * in / out) (resnet.py:156-159). */
int mdb_upsample_nearest(const void* x, int n, int h, int w, int c, void* out, int ho, int wo, void* stream);
/* nn.AdaptiveAvgPool2d((ho, wo)) over an NHWC fp32 map, optionally followed by SiLU: the pooling block of
 * BEVControlNetConditioningEmbeddingPlus (magicdrive/networks/map_embedder.py:118, forward :66-76 applies SiLU after every
 * block, the pool included).  Step-invariant (once per scene). */
int mdb_adaptive_avgpool(const float* x, int n, int h, int w, int c, float* out, int ho, int wo, int silu, void* stream);

/* Skinny linear for tiny M (time embedding MLP, time_emb_proj, camera / box encoders):
 * out[m, n] = act(in)[m, :] . W[n, :] + b[n], W bf16 [n, k] (ldw), in/out fp32.  pre_silu applies SiLU to the input,
 * post_silu to the output (embeddings.py:192-201; resnet.py:615-616; bbox_embedder.py:145-152). */
int mdb_linear_small(const float* in, int m, int k, int ldi, const void* w, int ldw, const float* bias, int n,
                     int pre_silu, int post_silu, float* out, int ldo, void* stream);

/* Sinusoidal timestep embedding, flip_sin_to_cos, freq_shift (embeddings.py:24-64).  t: fp32 [m] on device. */
int mdb_timestep_embedding(const float* t, int m, int dim, int flip_sin_to_cos, float freq_shift, float* out,
                           void* stream);

/* NeRF Fourier features [x, sin(2^k x), cos(2^k x)]_{k<num_freqs} on the last dim d of fp32 [rows, d]
 * (magicdrive/networks/embedder.py:15-40). out fp32 [rows, d*(1+2*num_freqs)]. */
int mdb_fourier_embed(const float* x, long long rows, int d, int num_freqs, float* out, void* stream);

/* dtype conversions / layout: NCHW fp32|bf16 <-> NHWC bf16 (pipeline boundary, pipeline_bev_controlnet.py:409-411). */
int mdb_nchw_to_nhwc(const void* x, int x_is_f32, int n, int c, int h, int w, void* out_bf16, void* stream);
int mdb_nhwc_to_nchw(const void* x_bf16, int n, int c, int h, int w, void* out, int out_is_f32, void* stream);
int mdb_f32_to_bf16(const float* x, void* out, long long n, void* stream);
int mdb_bf16_to_f32(const void* x, float* out, long long n, void* stream);

/* Latents [pix, cin] (fp32 or bf16) -> bf16 [repeat*pix, cpad] with channels >= cin zeroed: the K-padded A operand
 * that lets conv_in (unet_2d_condition.py:231, 4 -> 320 channels) run on the tensor-core path; repeat = 2 duplicates
 * the batch for classifier-free guidance (pipeline_bev_controlnet.py:352-354). */
int mdb_pack_latents(const void* x, int x_is_f32, long long pix, int cin, int cpad, int repeat, void* out, void* stream);

/* Image patches for the VAE encoder's conv_in (diffusers/models/vae.py:53-59, a 3x3 pad-1 nn.Conv2d from the cin = 3 image
 * channels; called from AutoencoderKL.encode, autoencoder_kl.py:164): NCHW images [n, cin, h, w] (fp32 or bf16) ->
 * bf16 [n*h*w, 64] where column (r*3 + s)*cin + c holds channel c at tap (r, s) of the zero-padded 3x3 neighbourhood and
 * columns >= 9*cin are zero (cin <= 7).  conv_in then runs as one K = 64 GEMM on mdb_gemm_conv with its weight packed in
 * the same column order, instead of a 9-tap conv over channels padded to 64.  out must be 16-byte aligned. */
int mdb_pack_image_patches(const void* x, int x_is_f32, int n, int cin, int h, int w, void* out, void* stream);

/* DiagonalGaussianDistribution of the encoder's moments (diffusers/models/vae.py:397-416; the demo's
 * `vae.encode(x).latent_dist.mean * scaling_factor`, demo/run_cond_on_view.py:80-86): moments fp32 NHWC [n*h*w, ldm] with
 * mean in columns [0, c) and logvar in [c, 2c) -> out fp32 NCHW [n, c, h, w] =
 *   scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)
 * noise: fp32 NCHW [n, c, h, w] (the shape randn_tensor draws in) or NULL, which gives scale * mean. */
int mdb_latent_dist(const float* moments, int ldm, int n, int c, int h, int w, const float* noise, float scale, float* out,
                    void* stream);

/* Classifier-free guidance + DDIM (eta = 0) update fused (pipeline_bev_controlnet.py:426-436;
 * scheduling_ddim.py:325-445).  eps: fp32 [(2 if cfg else 1) * n/c pixels, eps_ld] (uncond half first), c channels
 * used per pixel.  coef: device fp32[2] = {sqrt(abar_prev/abar_t), sqrt(1-abar_prev) - sqrt(abar_prev*(1-abar_t)/abar_t)}
 * so x_prev = c0*x + c1*eps.  latents: fp32 [n/c, c] updated in place. */
int mdb_cfg_ddim_step(const float* eps, int eps_ld, int c, int cfg, float guidance, const float* coef, float* latents,
                      long long n, void* stream);

/* Classifier-free guidance + one UniPCMultistepScheduler step fused (the reference's default sampler,
 * magicdrive/misc/test_utils.py:129; scheduling_unipc_multistep.py:518-600 with solver_order 2, bh2, predict_x0,
 * epsilon prediction).  eps as in mdb_cfg_ddim_step.  latents, last_sample, m0, m1: fp32 [n/c, c], all updated in
 * place (sample, sample before the last predictor, newest and previous x0 prediction; zero them before step 0).
 * coef: device fp32[12] for this step = {a0, a1, c0, c1, c2, c3, p0, p1, p2, use_corrector, 0, 0}:
 *   x0 = a0 x + a1 eps;  xc = use_corrector ? c0 last + c1 m0 + c2 m1 + c3 x0 : x;  x' = p0 xc + p1 x0 + p2 m0. */
int mdb_cfg_unipc_step(const float* eps, int eps_ld, int c, int cfg, float guidance, const float* coef, float* latents,
                       float* last_sample, float* m0, float* m1, long long n, void* stream);

/* Given-view generation (magicdrive/pipeline/pipeline_bev_controlnet_given_view.py:263-296, 379-389): for every view v
 * with view_mask[v] != 0, rows [v*rows_per_view, (v+1)*rows_per_view) of dst (fp32, row stride dst_ld, c channels used)
 * become coef[0]*a + coef[1]*b; a, b: fp32 [n_views*rows_per_view, c] contiguous, a may be NULL (term dropped);
 * coef: device fp32[2].  Used to re-noise pinned views (scheduler.add_noise) and to replace their predicted noise. */
int mdb_pin_views(float* dst, int dst_ld, const float* a, const float* b, int c, const float* coef, const int* view_mask,
                  long long rows_per_view, int n_views, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Input preparation (the step before the path; magicdrive/dataset/utils.py:120-352, demo/helper.py:386-466).
 * mdb_prepare_boxes: for every (scene, camera view) keep the boxes that have at least one corner in front of the camera
 * (z > 0 in the frame img_aug @ lidar2camera; the TEST uses the box shifted down by dz/2 exactly like the reference's
 * box_center_shift), compacted in their original order, as 8 corners (mmdet3d order) of the ORIGINAL box.
 *   boxes: fp32 [sum n_s, box_dim] rows (x, y, z, dx, dy, dz, yaw, ...), bottom-centred; labels: int64 [sum n_s];
 *   box_offsets: int32 [n_scenes + 1]; lidar2camera, img_aug (may be NULL): fp32 [n_scenes, n_views, 4, 4];
 *   out_boxes fp32 [n_scenes, n_views, capacity, 8, 3] (0-padded), out_classes int64 [.., capacity] (-1 padded),
 *   out_masks uint8 [.., capacity], out_counts int32 [n_scenes, n_views] (visible boxes, may exceed capacity: overflow is dropped).
 * mdb_camera_param: out fp32 [n, 3, 7] = [K[:3,:3] | (lidar2camera^-1)[:3]] for n = scenes * views rigid transforms
 * (dataset/utils.py:294-297). */
int mdb_prepare_boxes(const float* boxes, int box_dim, const long long* labels, const int* box_offsets, int n_scenes,
                      const float* lidar2camera, const float* img_aug, int n_views, int capacity, float* out_boxes,
                      long long* out_classes, unsigned char* out_masks, int* out_counts, void* stream);
int mdb_camera_param(const float* intrinsics, const float* lidar2camera, int n, float* out, void* stream);

/* Barrier between the `world` GPUs of a sharding group over NVLink peer memory, as one stream operation (graph-capturable).
 * flag_ptrs_dev: device array of `world` pointers, entry i = GPU i's symmetric uint32[n_channels * world] flag array as mapped
 * into THIS GPU's address space; epoch_dev: this GPU's uint32[n_channels] counter; timed_out_dev: int set to 1 if a peer did
 * not arrive within timeout_cycles SM cycles (0 = wait for ever).  Everything the peers wrote before their call is visible to
 * the kernels launched after this one (the view-sharded cross-view attention reads the neighbours' K/V right after it). */
int mdb_peer_barrier(void* const* flag_ptrs_dev, int rank, int world, int channel, int n_channels, void* epoch_dev,
                     long long timeout_cycles, int* timed_out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif
